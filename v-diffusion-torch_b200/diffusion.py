"""Drop-in for the sampling half of ``v_diffusion.diffusion`` (diffusion.py:42-112, 260-414).

``GaussianDiffusion.p_sample`` keeps the reference signature.  When ``denoise_fn`` is this
package's ``UNet`` the whole reverse loop runs inside the C library (one CUDA graph per step, the
v->x0 / clip / posterior mean / guidance combine / noise update fused in one kernel).  Any other
callable (e.g. a recording wrapper around the UNet) goes through the same fused update kernel one
step at a time, so tests can observe per-step model outputs.
"""
import ctypes as C
import math

import torch

from . import _lib
from .unet import UNet


class LogSNRSchedule:
    """Callable returned by get_logsnr_schedule; also carries the parameters the C side needs."""

    def __init__(self, schedule, logsnr_min, logsnr_max):
        if schedule not in _lib.SCHEDULES:
            raise NotImplementedError(schedule)                     # diffusion.py:96
        self.schedule, self.logsnr_min, self.logsnr_max = schedule, float(logsnr_min), float(logsnr_max)

    def __call__(self, t):
        tt = t.to(torch.float64)
        lmin, lmax = self.logsnr_min, self.logsnr_max
        if self.schedule == "cosine":
            a = math.atan(math.exp(-0.5 * lmax)) / (0.5 * math.pi)
            b = math.atan(math.exp(-0.5 * lmin)) / (0.5 * math.pi)
            out = -2 * torch.log(torch.tan((a + tt * (b - a)) * math.pi * 0.5))
        elif self.schedule == "linear":
            a, b = 1 / (1 + math.exp(-lmax)), 1 / (1 + math.exp(-lmin))
            out = torch.logit(a + tt * (b - a))
        elif self.schedule == "sigmoid":
            out = lmax - tt * (lmax - lmin)
        else:
            x_to = 0.9999 + tt * (0.98 - 0.9999)
            la = 1000 / -0.0199 * (x_to * torch.log(x_to) - x_to - 0.9999 * math.log(0.9999) + 0.9999)
            z = la - 1e-9
            out = la - torch.where(z < -9, torch.log1p(-torch.exp(z)), torch.log(-torch.expm1(z)))
        return out.to(t.dtype)


def get_logsnr_schedule(schedule, logsnr_min: float = -20., logsnr_max: float = 20., rescale: bool = False):
    if rescale:
        raise NotImplementedError("allow_rescale is off in every reference config (defaults.json:45)")
    return LogSNRSchedule(schedule, logsnr_min, logsnr_max)


class GaussianDiffusion:
    def __init__(self, logsnr_fn, sample_timesteps, model_out_type, model_var_type, reweight_type, loss_type,
                 intp_frac=None, w_guide=0.1, p_uncond=0.1, x0eps_coef=False):
        if not isinstance(logsnr_fn, LogSNRSchedule):
            raise TypeError("logsnr_fn must come from v_diffusion_b200.get_logsnr_schedule")
        if model_out_type not in _lib.OUT_TYPES:
            raise NotImplementedError(model_out_type)               # diffusion.py:253-257
        self.logsnr_fn = logsnr_fn
        self.sample_timesteps = sample_timesteps
        self.model_out_type, self.model_var_type = model_out_type, model_var_type
        self.reweight_type, self.loss_type = reweight_type, loss_type
        self.intp_frac, self.w_guide, self.p_uncond, self.x0eps_coef = intp_frac, w_guide, p_uncond, x0eps_coef

    # ------------------------------------------------------------------ C structs
    def _check_solver(self, solver, use_ddim):
        """``solver`` (extension): None, the reference's first-order step, or "dpmpp_2m", DPM-Solver++(2M) (Lu et al., 2022)
        on the same time grid -- defined for DDIM (use_ddim=True) with x0eps_coef=False only."""
        if solver not in _lib.SOLVERS:
            raise NotImplementedError(f"unknown solver {solver!r} (choices: None, 'dpmpp_2m')")
        if solver is not None and not use_ddim:
            raise NotImplementedError(f"solver={solver!r} needs use_ddim=True (it is not defined for ancestral sampling)")
        if solver is not None and self.x0eps_coef:
            raise NotImplementedError(f"solver={solver!r} needs x0eps_coef=False (under DDIM the reference's (eps, x0) "
                                      "coefficients are logarithms, diffusion.py:180-182)")

    def sampler_config(self, use_ddim, seed=None, t_fp32=False, solver=None):
        self._check_solver(solver, use_ddim)
        if not use_ddim and self.model_var_type not in _lib.VAR_TYPES:
            raise NotImplementedError(self.model_var_type)          # diffusion.py:161
        if not use_ddim and self.model_var_type == "fixed_medium" and not isinstance(self.intp_frac, float):
            raise AssertionError("fixed_medium needs a float intp_frac")   # diffusion.py:155
        sc = _lib.SamplerConfig()
        sc.sample_timesteps = int(self.sample_timesteps)
        sc.model_out_type = _lib.OUT_TYPES[self.model_out_type]
        sc.model_var_type = _lib.VAR_TYPES.get(self.model_var_type, 1)
        sc.logsnr_schedule = _lib.SCHEDULES[self.logsnr_fn.schedule]
        sc.use_ddim = int(bool(use_ddim))
        sc.x0eps_coef = int(bool(self.x0eps_coef))                  # diffusion.py:137-140, 180-182, 335-343
        sc.t_fp32 = int(bool(t_fp32))                               # diffusion.py:421 vs :399
        sc.solver = _lib.SOLVERS[solver]
        sc.intp_frac = float(self.intp_frac or 0.)
        sc.logsnr_min, sc.logsnr_max = self.logsnr_fn.logsnr_min, self.logsnr_fn.logsnr_max
        sc.w_guide = float(self.w_guide)
        sc.seed = int(seed or 0) & (2 ** 64 - 1)
        return sc

    @staticmethod
    def _noise_seed(seed):
        """Seed of the on-device noise stream of one call.  ``seed=None`` in the reference means "draw from the global
        generator" (diffusion.py:401-402), i.e. fresh noise on every call; here a fresh 63-bit seed is drawn from
        torch's global CPU generator, so repeated calls differ and ``torch.manual_seed`` still makes a run repeatable."""
        if seed is not None:
            return int(seed)
        return int(torch.randint(0, 2 ** 63 - 1, (1,), dtype=torch.int64).item())

    @staticmethod
    def _prepare_label(denoise_fn, label, B, device):
        """Labels as the C side reads them: int64 (B,) class ids in [0, num_classes] (0 = no class), or fp32 multi-hot
        (B, num_classes) rows for a multitag UNet (unet.py:290-294).  Shapes and ranges are checked here because the
        library only sees raw pointers (the reference's F.one_hot raises on an out-of-range id, modules.py:191-196)."""
        if label is None:
            return None
        multitags = bool(getattr(denoise_fn, "multitags", False)) or label.ndim == 2   # (a wrapped UNet hides its flag)
        num_classes = int(getattr(denoise_fn, "num_classes", 0) or 0)
        label = label.to(device=device, dtype=torch.float32 if multitags else torch.int64).contiguous()
        if isinstance(denoise_fn, UNet) and num_classes > 0:
            if multitags:
                if tuple(label.shape) != (B, num_classes):
                    raise ValueError(f"multitag labels must have shape ({B}, {num_classes}), got {tuple(label.shape)}")
            else:
                if label.numel() != B:
                    raise ValueError(f"labels must have one class id per sample ({B}), got shape {tuple(label.shape)}")
                label = label.reshape(B)
                lo, hi = int(label.min()), int(label.max())
                if lo < 0 or hi > num_classes:
                    raise RuntimeError(f"class ids must lie in [0, {num_classes}] (0 = unconditional), got [{lo}, {hi}]")
        return label

    def _check_inpaint(self, shape, known, mask, known_noise):
        """Inpainting inputs (extension; include/vdt_b200.h vdt_inpaint) as fp32 tensors on the caller's devices, or None when
        there are none.  ``known``: the image in model space, shaped like the batch; ``mask``: 1 = known pixel, values in
        [0, 1], shaped like the batch or (B, 1, R, R); ``known_noise``: optional (T,) + shape draws of z'.  Everything is
        checked here because the library only sees raw pointers; the value checks share one device synchronisation."""
        if known is None and mask is None:
            if known_noise is not None:
                raise ValueError("known_noise needs known and mask")
            return None
        if (known is None) != (mask is None):
            raise ValueError("inpainting needs both known and mask")
        shape = tuple(shape)
        if tuple(known.shape) != shape:
            raise ValueError(f"known has shape {tuple(known.shape)}, expected {shape}")
        if tuple(mask.shape) not in (shape, shape[:1] + (1,) + shape[2:]):
            raise ValueError(f"mask has shape {tuple(mask.shape)}, expected {shape} or {shape[:1] + (1,) + shape[2:]}")
        if known_noise is not None and tuple(known_noise.shape) != (self.sample_timesteps,) + shape:
            raise ValueError(f"known_noise has shape {tuple(known_noise.shape)}, expected {(self.sample_timesteps,) + shape}")
        known, mask = known.to(torch.float32), mask.to(torch.float32)
        flags = [torch.isfinite(known).all(), ((mask >= 0) & (mask <= 1)).all()]
        if known_noise is not None:
            known_noise = known_noise.to(torch.float32)
            flags.append(torch.isfinite(known_noise).all())
        ok = torch.stack([f.to(known.device) for f in flags]).tolist()
        if not ok[0]:
            raise ValueError("known must be finite")
        if not ok[1]:
            raise ValueError("mask values must lie in [0, 1]")
        if known_noise is not None and not ok[2]:
            raise ValueError("known_noise must be finite")
        return known, mask, known_noise

    @staticmethod
    def _inpaint_on(inp, shape, device):
        """The checked inputs as contiguous device tensors (the mask expanded over channels) and their vdt_inpaint struct."""
        known, mask, known_noise = inp
        known = known.to(device).contiguous()
        mask = mask.to(device).expand(tuple(shape)).contiguous()
        known_noise = None if known_noise is None else known_noise.to(device).contiguous()
        return (known, mask, known_noise), _lib.Inpaint(_lib.ptr(known), _lib.ptr(mask), _lib.ptr(known_noise))

    def step_coefficients(self, use_ddim, solver=None):
        """[T, 16] fp32 host table (include/vdt_b200.h: vdt_step_coefficients); slot 15 holds DPM-Solver++(2M)'s c2k."""
        sc = self.sampler_config(use_ddim, solver=solver)
        out = torch.empty((self.sample_timesteps, _lib.COEF_STRIDE), dtype=torch.float32)
        _lib.check(_lib.lib().vdt_step_coefficients(C.byref(sc), _lib.ptr(out)))
        return out

    def invert_coefficients(self):
        """[T, 16] fp32 host table of DDIM inversion (include/vdt_b200.h: vdt_invert_coefficients): row j maps x at j/T to
        x at (j+1)/T."""
        self._check_invertible()
        sc = self.sampler_config(True)
        out = torch.empty((self.sample_timesteps, _lib.COEF_STRIDE), dtype=torch.float32)
        _lib.check(_lib.lib().vdt_invert_coefficients(C.byref(sc), _lib.ptr(out)))
        return out

    def _check_invertible(self):
        if self.x0eps_coef:
            raise NotImplementedError("DDIM inversion needs x0eps_coef=False (under DDIM the reference's (eps, x0) "
                                      "coefficients are logarithms, diffusion.py:180-182)")

    def _check_start_step(self, start_step):
        """``start_step`` k of p_sample: None means T (a whole trajectory), else an int in [1, T]."""
        T = self.sample_timesteps
        if start_step is None:
            return T
        if isinstance(start_step, bool) or not isinstance(start_step, int) or not 1 <= start_step <= T:
            raise ValueError(f"start_step must be an int in [1, {T}] (x is given at t = start_step / T), got {start_step!r}")
        return start_step

    # ------------------------------------------------------------------ p_sample (diffusion.py:394-414)
    @torch.no_grad()
    def p_sample(self, denoise_fn, shape, noise=None, label=None, device="cpu", seed=None, use_ddim=False,
                 step_noise=None, solver=None, known=None, mask=None, known_noise=None, start_step=None):
        """``step_noise`` (extension): optional (T, B, C, H, W) tensor of the per-step normal draws the
        reference takes from its generator (diffusion.py:389), so both sides inject identical noise.
        ``solver`` (extension): None (the reference's step) or "dpmpp_2m" (DPM-Solver++(2M), with use_ddim=True).
        ``known``, ``mask``, ``known_noise`` (extension): inpainting by replacement.  After every step the pixels with mask 1
        are set to ``known`` diffused to the step's time (alpha_s known + sigma_s z'), and the last step sets them to ``known``;
        a soft mask blends.  z' comes from ``known_noise`` or else from the library's noise stream keyed by ``seed`` (a fresh
        seed when None, under DDIM too).  See include/vdt_b200.h vdt_inpaint.
        ``start_step`` (extension): k in [1, T]; ``noise`` is then x at t = k/T (e.g. an inverted latent, or an image diffused
        to k/T for SDEdit) and steps k-1 ... 0 run as a fresh trajectory (DPM-Solver++(2M) starts first-order).  None means T,
        the reference's loop.  ``step_noise`` and ``known_noise`` keep their (T, ...) shapes, indexed by step."""
        self._check_solver(solver, use_ddim)
        inp = self._check_inpaint(shape, known, mask, known_noise)
        k = self._check_start_step(start_step)
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("v_diffusion_b200 samples on CUDA (sm_100a) only; there is no CPU fallback")
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        B = shape[0]
        gen = None if seed is None else torch.Generator(device).manual_seed(seed)
        if noise is None:
            x_t = torch.randn(shape, device=device, generator=gen)
        else:
            x_t = noise.to(device)
        x_t = x_t.to(torch.float32).contiguous()
        if tuple(x_t.shape) != tuple(shape):
            raise ValueError(f"noise has shape {tuple(x_t.shape)}, expected {tuple(shape)}")
        if B == 0:                                           # an empty batch has nothing to launch
            return x_t.cpu()
        label = self._prepare_label(denoise_fn, label, B, device)
        if step_noise is not None:
            step_noise = step_noise.to(device=device, dtype=torch.float32).contiguous()
            if tuple(step_noise.shape) != (self.sample_timesteps,) + tuple(shape):
                raise ValueError(f"step_noise must have shape {(self.sample_timesteps,) + tuple(shape)}")
        L = _lib.lib()
        # inpainting without injected z' draws it from the library's stream keyed by the call's seed, under DDIM too
        inp_seed = inp is not None and known_noise is None
        if isinstance(denoise_fn, UNet):
            # fused path: the per-step normals come from the library's own Philox stream keyed by this call's seed
            sc = self.sampler_config(use_ddim, self._noise_seed(seed) if ((not use_ddim and step_noise is None) or inp_seed)
                                     else seed, solver=solver)
            plan = denoise_fn.plan_for(shape[2], device)
            out = torch.empty_like(x_t)
            with torch.cuda.device(device):
                if start_step is not None:
                    held, ip = self._inpaint_on(inp, shape, device) if inp is not None else (None, None)   # kept alive
                    out.copy_(x_t)
                    _lib.check(L.vdt_p_sample_from(plan, C.byref(sc), None if ip is None else C.byref(ip), _lib.ptr(out),
                                                   _lib.ptr(label), _lib.ptr(step_noise), B, k - 1, _lib.current_stream_ptr()))
                elif inp is None:
                    _lib.check(L.vdt_p_sample(plan, C.byref(sc), _lib.ptr(x_t), _lib.ptr(label), _lib.ptr(step_noise),
                                              _lib.ptr(out), B, _lib.current_stream_ptr()))
                else:
                    held, ip = self._inpaint_on(inp, shape, device)      # `held` keeps the tensors alive for the call
                    _lib.check(L.vdt_p_sample_inpaint(plan, C.byref(sc), C.byref(ip), _lib.ptr(x_t), _lib.ptr(label),
                                                      _lib.ptr(step_noise), _lib.ptr(out), B, _lib.current_stream_ptr()))
            return out.cpu()
        # generic callable: same fused update kernel, one step at a time; the per-step normals continue the generator
        # that produced x_T, like the reference's single generator (diffusion.py:401-405, 389)
        sc = self.sampler_config(use_ddim, self._noise_seed(seed) if inp_seed else seed, solver=solver)
        held = None if inp is None else self._inpaint_on(inp, shape, device)[0]
        return self._p_sample_generic(denoise_fn, shape, x_t, label, step_noise, sc, device, gen, use_ddim, solver, held, k).cpu()

    @torch.no_grad()
    def p_sample_progressive(self, denoise_fn, shape, noise=None, label=None, device="cpu", seed=None, use_ddim=False,
                             pred_freq=50, step_noise=None, solver=None, known=None, mask=None, known_noise=None):
        """diffusion.py:416-441: returns (x_0, preds) where preds[k] is the (guided) x0 prediction made at the
        steps ti with (ti + 1) % pred_freq == 0, ordered like the reference (index L-1 = earliest).  Fused path only.
        ``solver`` as in p_sample; under "dpmpp_2m" the ``pred`` buffer every range call shares carries the previous
        step's guided x0 into the next call.  ``known``, ``mask``, ``known_noise`` as in p_sample; the previews stay the
        model's guided x0 predictions."""
        self._check_solver(solver, use_ddim)
        inp = self._check_inpaint(shape, known, mask, known_noise)
        if not isinstance(denoise_fn, UNet):
            raise TypeError("p_sample_progressive needs the v_diffusion_b200 UNet")
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("v_diffusion_b200 samples on CUDA (sm_100a) only; there is no CPU fallback")
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        B, T = shape[0], self.sample_timesteps
        gen = None if seed is None else torch.Generator(device).manual_seed(seed)
        x = (torch.randn(shape, device=device, generator=gen) if noise is None else noise.to(device)).to(torch.float32).contiguous().clone()
        label = self._prepare_label(denoise_fn, label, B, device)
        if step_noise is not None:
            step_noise = step_noise.to(device=device, dtype=torch.float32).contiguous()
        # the reference's progressive loop carries an fp32 step tensor (diffusion.py:421): fp32 s / t and an fp32 sinusoid
        inp_seed = inp is not None and known_noise is None
        sc = self.sampler_config(use_ddim, self._noise_seed(seed) if ((not use_ddim and step_noise is None) or inp_seed) else seed,
                                 t_fp32=True, solver=solver)
        held, ip = self._inpaint_on(inp, shape, device) if inp is not None else (None, None)   # `held` keeps them alive
        plan = denoise_fn.plan_for(shape[2], device)
        Lp = T // pred_freq
        preds = torch.zeros((Lp, B) + tuple(shape[1:]), dtype=torch.float32)
        pred = torch.empty_like(x)
        lib, idx, first = _lib.lib(), Lp, T - 1
        with torch.cuda.device(device):
            while first >= 0:
                # run down to (and including) the next step whose prediction is recorded: (ti + 1) % pred_freq == 0
                stop = ((first + 1) // pred_freq) * pred_freq - 1
                record = stop >= 0
                if not record:
                    stop = 0
                if ip is None:
                    _lib.check(lib.vdt_p_sample_range(plan, C.byref(sc), _lib.ptr(x), _lib.ptr(label), _lib.ptr(step_noise), B,
                                                      first, first - stop + 1, _lib.ptr(pred), _lib.current_stream_ptr()))
                else:
                    _lib.check(lib.vdt_p_sample_range_inpaint(plan, C.byref(sc), C.byref(ip), _lib.ptr(x), _lib.ptr(label),
                                                              _lib.ptr(step_noise), B, first, first - stop + 1, _lib.ptr(pred),
                                                              _lib.current_stream_ptr()))
                if record and idx > 0:
                    idx -= 1
                    preds[idx] = pred.cpu()
                first = stop - 1
        return x.cpu(), preds

    # ------------------------------------------------------------------ DDIM inversion (extension)
    @torch.no_grad()
    def ddim_invert(self, denoise_fn, x_0, label=None, device="cuda", num_steps=None, w_guide=None):
        """DDIM inversion (Song et al., DDIM, section 4.3): runs the deterministic DDIM ODE forward in time from the image
        ``x_0`` (model space, (B, C, R, R)) and returns x at t = num_steps / T on the CPU, like p_sample.  ``num_steps=None``
        means T (a full encoding); ``p_sample(..., noise=latent, start_step=num_steps, use_ddim=True)`` decodes it again.
        Step j evaluates the model at j/T and uses its unclipped x0; under CFG (``w_guide`` > 0 and labels, ``w_guide=None``
        meaning ``self.w_guide``) the guided x0c + w (x0c - x0u).  The UNet runs on the fused path; any other callable goes
        one step at a time through vdt_op_invert_step.  See include/vdt_b200.h vdt_ddim_invert_range.

        For an "x0" model the first step multiplies the model's error at t = 0 by sigma_t / sigma_s (about 350 at T = 100 on
        the cosine +-20 schedule), so an untrained x0 network's latents grow large; "v", "eps" and "both" are benign there."""
        self._check_invertible()
        T = self.sample_timesteps
        n = T if num_steps is None else num_steps
        if isinstance(n, bool) or not isinstance(n, int) or not 0 <= n <= T:
            raise ValueError(f"num_steps must be an int in [0, {T}], got {num_steps!r}")
        w = float(self.w_guide if w_guide is None else w_guide)
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("v_diffusion_b200 samples on CUDA (sm_100a) only; there is no CPU fallback")
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        x = x_0.to(device=device, dtype=torch.float32).contiguous().clone()
        if x.ndim != 4:
            raise ValueError(f"x_0 must have shape (B, C, R, R), got {tuple(x.shape)}")
        B = x.shape[0]
        if B == 0 or n == 0:
            return x.cpu()
        label = self._prepare_label(denoise_fn, label, B, device)
        sc = self.sampler_config(True)
        sc.w_guide = w
        L = _lib.lib()
        with torch.cuda.device(device):
            if isinstance(denoise_fn, UNet):
                plan = denoise_fn.plan_for(x.shape[2], device)
                _lib.check(L.vdt_ddim_invert_range(plan, C.byref(sc), _lib.ptr(x), _lib.ptr(label), B, 0, n,
                                                   _lib.current_stream_ptr()))
                return x.cpu()
            coefs = self.invert_coefficients()
            use_cfg = (w > 0) and (label is not None)              # the sampler's rule (diffusion.py:368)
            hw = x.shape[2] * x.shape[3]
            for j in range(n):
                t = torch.full((B,), j / T, dtype=torch.float64, device=device)
                if use_cfg:
                    xin, tin = x.repeat_interleave(2, dim=0), t.repeat_interleave(2)
                    yin = label.repeat_interleave(2, dim=0)
                    yin[1::2] = 0
                else:
                    xin, tin, yin = x, t, label
                model_out = denoise_fn(xin, tin, yin).to(torch.float32).contiguous()
                x_next = torch.empty_like(x)
                _lib.check(L.vdt_op_invert_step(_lib.ptr(model_out), _lib.ptr(x), _lib.ptr(x_next), B, x.shape[1], hw,
                                                int(use_cfg), sc.model_out_type, _lib.ptr(coefs[j].contiguous()), w,
                                                _lib.current_stream_ptr()))
                x = x_next
        return x.cpu()

    # ------------------------------------------------------------------ likelihood in bits/dim (extension)
    def _check_bpd(self):
        if self.x0eps_coef:
            raise NotImplementedError("the likelihood bound needs x0eps_coef=False (the reference's (eps, x0) posterior "
                                      "coefficients are another parameterisation of the mean, and under DDIM logarithms)")
        if self.model_var_type not in _lib.VAR_TYPES:
            raise NotImplementedError(f"the likelihood bound needs a fixed model_var_type, got {self.model_var_type!r}")

    def bpd_coefficients(self):
        """[T, 16] fp32 host table of the likelihood bound (include/vdt_b200.h: vdt_bpd_coefficients): the ancestral row of
        step i with slot 14 = K_i and slot 15 = k_i, term_i = K_i + k_i mse_i for i > 0."""
        self._check_bpd()
        sc = self.sampler_config(False)
        out = torch.empty((self.sample_timesteps, _lib.COEF_STRIDE), dtype=torch.float32)
        _lib.check(_lib.lib().vdt_bpd_coefficients(C.byref(sc), _lib.ptr(out)))
        return out

    @torch.no_grad()
    def calc_all_bpd(self, denoise_fn, x_0, y=None, clip_denoised=True, device="cuda", seed=None, noise=None):
        """Negative ELBO in bits per dimension of the images ``x_0`` (model space [-1, 1], (B, C, R, R)), the standard
        variational bound of Ho et al. (2020, section 3.3) as Nichol & Dhariwal's calc_bpd_loop computes it, on this
        library's time grid t = (i+1)/T and coefficient table.  The definition is written out in include/vdt_b200.h
        (vdt_calc_bpd_range); it is not pinned to the reference's own likelihood code, and the name and return layout follow
        the reference family without its exact signature having been checked.

        Returns ``(total_bpd [B], terms_bpd [B, T], prior_bpd [B], mse [B, T])``, fp64 on the CPU: term i is the KL of step i
        (i > 0) or the 8-bit decoder's negative log-likelihood (i = 0), mse[:, i] the mean squared error of the (clipped iff
        ``clip_denoised``) x0 prediction, and total = terms.sum(1) + prior.  ``y``: labels as in p_sample; guidance plays no
        part.  The q-sample draws eps_i come from ``noise`` ((T, B, C, R, R), indexed by step) or else from a stream keyed by
        ``seed`` (a fresh seed when None): the library's own on the fused path (the UNet), a torch generator for any other
        callable, which runs one step at a time through vdt_op_bpd_term."""
        self._check_bpd()
        T = self.sample_timesteps
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("v_diffusion_b200 evaluates on CUDA (sm_100a) only; there is no CPU fallback")
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        x0 = x_0.to(device=device, dtype=torch.float32).contiguous()
        if x0.ndim != 4 or x0.shape[2] != x0.shape[3]:
            raise ValueError(f"x_0 must have shape (B, C, R, R), got {tuple(x0.shape)}")
        B, Cc, R = x0.shape[0], x0.shape[1], x0.shape[2]
        if noise is not None:
            noise = noise.to(device=device, dtype=torch.float32).contiguous()
            if tuple(noise.shape) != (T,) + tuple(x0.shape):
                raise ValueError(f"noise has shape {tuple(noise.shape)}, expected {(T,) + tuple(x0.shape)}")
        if B == 0:
            return (torch.zeros(0, dtype=torch.float64), torch.zeros((0, T), dtype=torch.float64),
                    torch.zeros(0, dtype=torch.float64), torch.zeros((0, T), dtype=torch.float64))
        flags = [torch.isfinite(x0).all()] + ([torch.isfinite(noise).all()] if noise is not None else [])
        ok = torch.stack(flags).tolist()
        if not ok[0]:
            raise ValueError("x_0 must be finite")
        if noise is not None and not ok[1]:
            raise ValueError("noise must be finite")
        label = self._prepare_label(denoise_fn, y, B, device)
        sc = self.sampler_config(False, self._noise_seed(seed) if noise is None else seed)
        terms = torch.empty((B, T), dtype=torch.float64, device=device)
        mse = torch.empty((B, T), dtype=torch.float64, device=device)
        prior = torch.empty((B,), dtype=torch.float64, device=device)
        chw, clip = Cc * R * R, int(bool(clip_denoised))
        L = _lib.lib()
        with torch.cuda.device(device):
            _lib.check(L.vdt_bpd_prior(C.byref(sc), _lib.ptr(x0), B, chw, _lib.ptr(prior), _lib.current_stream_ptr()))
            if isinstance(denoise_fn, UNet):
                plan = denoise_fn.plan_for(R, device)
                _lib.check(L.vdt_calc_bpd_range(plan, C.byref(sc), _lib.ptr(x0), _lib.ptr(label), _lib.ptr(noise), clip, B, 0, T,
                                                _lib.ptr(terms), _lib.ptr(mse), _lib.current_stream_ptr()))
            else:
                coefs = self.bpd_coefficients()
                coef_dev = coefs.to(device)
                gen = torch.Generator(device).manual_seed(sc.seed) if noise is None else None
                want = (B, (2 if self.model_out_type == "both" else 1) * Cc, R, R)
                for i in reversed(range(T)):                   # the fused path's order (and the generator's)
                    eps = noise[i] if noise is not None else torch.randn(tuple(x0.shape), device=device, generator=gen)
                    x_t = torch.empty_like(x0)
                    _lib.check(L.vdt_q_sample(_lib.ptr(x0), _lib.ptr(eps), _lib.ptr(coef_dev[i].expand(B, -1).contiguous()),
                                              _lib.ptr(x_t), B, chw, _lib.current_stream_ptr()))
                    t = torch.full((B,), (i + 1) / T, dtype=torch.float64, device=device)
                    out = denoise_fn(x_t, t, label).to(torch.float32).contiguous()
                    if tuple(out.shape) != want:
                        raise ValueError(f"model output has shape {tuple(out.shape)}, expected {want}")
                    _lib.check(L.vdt_op_bpd_term(_lib.ptr(out), _lib.ptr(x_t), _lib.ptr(x0), B, Cc, R * R, sc.model_out_type, i, T,
                                                 _lib.ptr(coefs[i].contiguous()), clip, _lib.ptr(terms), _lib.ptr(mse),
                                                 _lib.current_stream_ptr()))
        terms, mse, prior = terms.cpu(), mse.cpu(), prior.cpu()
        return terms.sum(dim=1) + prior, terms, prior, mse

    # ------------------------------------------------------------------ train_loss (diffusion.py:492-545)
    @torch.no_grad()
    def train_loss(self, denoise_fn, x_0, t, y, noise=None, return_grad=False):
        """Forward half of the training step around the model call (SURVEY §8 f2): q_sample, the model
        call, from_model_out_to_pred and the re-weighted MSE, as two fused kernels.  Returns the per-sample loss (B,) on
        x_0's device; with ``return_grad`` also d loss.mean() / d model_out -- the tensor the reference's autograd hands
        to the UNet's backward pass (training.TrainingStep passes its UNetTrainGraph as ``denoise_fn`` and feeds this gradient to the graph's backward).

        Reproduced as is: the label-dropout mask of ``p_uncond`` is applied to ``y`` in place AFTER the model call
        (diffusion.py:527-529 vs :508), so it changes the caller's tensor but never the loss; single-target reweightings
        compare the target with the raw model output (:541)."""
        if self.loss_type != "mse":
            raise NotImplementedError("loss_type 'kl' (likelihood evaluation, diffusion.py:446-464) is out of scope")
        if self.model_var_type == "learned":
            raise AssertionError("mse loss needs a fixed variance type")          # diffusion.py:519
        if self.reweight_type not in _lib.REWEIGHT_TYPES:
            raise AssertionError(self.reweight_type)                              # diffusion.py:520
        if x_0.device.type != "cuda":
            raise RuntimeError("v_diffusion_b200 trains on CUDA (sm_100a) only; there is no CPU fallback")
        dev = x_0.device
        B = x_0.shape[0]
        x_0 = x_0.to(torch.float32).contiguous()
        noise = torch.randn_like(x_0) if noise is None else noise.to(device=dev, dtype=torch.float32).contiguous()
        L = _lib.lib()
        sc = self.sampler_config(use_ddim=True)
        t_host = t.detach().to(device="cpu", dtype=torch.float64).reshape(-1).contiguous()
        if t_host.numel() != B:
            raise ValueError("t must have one entry per sample")
        coef_h = torch.empty((B, _lib.COEF_STRIDE), dtype=torch.float32)
        _lib.check(L.vdt_train_coefficients(C.byref(sc), _lib.ptr(t_host), B, _lib.ptr(coef_h)))
        coef = coef_h.to(dev)
        x_t = torch.empty_like(x_0)
        chw = x_0[0].numel()
        with torch.cuda.device(dev):
            _lib.check(L.vdt_q_sample(_lib.ptr(x_0), _lib.ptr(noise), _lib.ptr(coef), _lib.ptr(x_t), B, chw, _lib.current_stream_ptr()))
        model_out = denoise_fn(x_t, t, y).to(torch.float32).contiguous()
        if self.p_uncond and y is not None:                                        # diffusion.py:527-529: after the model call
            keep = torch.rand((y.shape[0],)) > self.p_uncond
            y *= keep.to(device=y.device, dtype=y.dtype).reshape((-1,) + (1,) * (y.ndim - 1))
        Cc, hw = x_0.shape[1], x_0.shape[2] * x_0.shape[3]
        want = (2 if self.model_out_type == "both" else 1) * Cc
        if model_out.shape != (B, want) + tuple(x_0.shape[2:]):
            raise ValueError(f"model output has shape {tuple(model_out.shape)}, expected {(B, want) + tuple(x_0.shape[2:])}")
        loss = torch.empty((B,), dtype=torch.float32, device=dev)
        grad = torch.empty_like(model_out) if return_grad else None
        with torch.cuda.device(dev):
            _lib.check(L.vdt_train_loss(_lib.ptr(model_out), _lib.ptr(x_0), _lib.ptr(noise), _lib.ptr(x_t), _lib.ptr(coef),
                                        _lib.ptr(loss), _lib.ptr(grad), B, Cc, hw, _lib.OUT_TYPES[self.model_out_type],
                                        _lib.REWEIGHT_TYPES[self.reweight_type], _lib.current_stream_ptr()))
        return (loss, grad) if return_grad else loss

    # ------------------------------------------------------------------ progressive distillation (extension)
    def distill_coefficients(self, step):
        """[2, B, 16] fp32 host table of progressive distillation (include/vdt_b200.h: vdt_distill_coefficients) for the
        student step indices ``step`` (B,) in [0, sample_timesteps): plane 0 at t = (i+1)/N, plane 1 at t' = (2i+1)/(2N)."""
        step_host = torch.as_tensor(step).detach().to(device="cpu", dtype=torch.int32).reshape(-1).contiguous()
        sc = self.sampler_config(use_ddim=True)
        out = torch.empty((2, step_host.numel(), _lib.COEF_STRIDE), dtype=torch.float32)
        _lib.check(_lib.lib().vdt_distill_coefficients(C.byref(sc), _lib.ptr(step_host), step_host.numel(), _lib.ptr(out)))
        return out

    @staticmethod
    def _teacher_rows(z, t, y, use_cfg):
        """The sampler's CFG layout (diffusion.py:368-372): rows 2b conditional, 2b+1 unconditional."""
        if not use_cfg:
            return z, t, y
        yin = y.repeat_interleave(2, dim=0)
        yin[1::2] = 0
        return z.repeat_interleave(2, dim=0), t.repeat_interleave(2), yin

    @torch.no_grad()
    def distill_loss(self, teacher_fn, student_fn, x_0, step, y, noise=None, w_guide=0., return_grad=False):
        """Progressive distillation (Salimans & Ho, 2022, Algorithm 2; include/vdt_b200.h vdt_distill_coefficients): the
        student, sampled with N = ``self.sample_timesteps`` DDIM steps, learns in one step from t = (i+1)/N to t'' = i/N what
        the teacher does in two DDIM steps on the 2N grid.  ``step``: the student step index i per sample, (B,) in [0, N).

        q_sample at t -> teacher at t -> vdt_op_distill_step (z_t', x1) -> teacher at t' -> vdt_op_distill_target (x~, eps~) ->
        student at t -> vdt_train_loss with x~ and eps~ as the targets, so every model_out_type and reweight_type works as in
        train_loss.  The teacher runs with CFG (2B interleaved rows) when ``w_guide`` > 0 and labels are given; the student
        sees the labels as given.  Both networks may be any callable ``(x, t, y) -> output``.  Returns the per-sample loss (B,)
        and, with ``return_grad``, d loss.mean() / d student output."""
        if self.loss_type != "mse":
            raise NotImplementedError("distillation trains with the mse loss")
        if self.model_var_type == "learned":
            raise AssertionError("mse loss needs a fixed variance type")
        if self.reweight_type not in _lib.REWEIGHT_TYPES:
            raise AssertionError(self.reweight_type)
        if x_0.device.type != "cuda":
            raise RuntimeError("v_diffusion_b200 trains on CUDA (sm_100a) only; there is no CPU fallback")
        if x_0.ndim != 4:
            raise ValueError(f"x_0 must have shape (B, C, H, W), got {tuple(x_0.shape)}")
        dev, B, N = x_0.device, x_0.shape[0], int(self.sample_timesteps)
        x_0 = x_0.to(torch.float32).contiguous()
        noise = torch.randn_like(x_0) if noise is None else noise.to(device=dev, dtype=torch.float32).contiguous()
        if noise.shape != x_0.shape:
            raise ValueError(f"noise has shape {tuple(noise.shape)}, expected {tuple(x_0.shape)}")
        step = torch.as_tensor(step).reshape(-1)
        if step.numel() != B:
            raise ValueError("step must have one entry per sample")
        coef = self.distill_coefficients(step).to(dev)                 # refuses steps outside [0, N)
        step = step.to(device=dev, dtype=torch.float64)
        t = (step + 1) / N                                              # the sampler's t at N, fp64
        t_mid = (2 * step + 1) / (2 * N)                                # its t at 2N
        w = float(w_guide)
        use_cfg = w > 0 and y is not None
        out_type = _lib.OUT_TYPES[self.model_out_type]
        Cc, hw = x_0.shape[1], x_0.shape[2] * x_0.shape[3]
        Cm = (2 if self.model_out_type == "both" else 1) * Cc
        L = _lib.lib()
        if y is not None:
            y = y.to(dev)

        def teacher(z, tt):
            out = teacher_fn(*self._teacher_rows(z, tt, y, use_cfg)).to(torch.float32).contiguous()
            want = (B * (2 if use_cfg else 1), Cm) + tuple(x_0.shape[2:])
            if tuple(out.shape) != want:
                raise ValueError(f"teacher output has shape {tuple(out.shape)}, expected {want}")
            return out

        z_t = torch.empty_like(x_0)
        with torch.cuda.device(dev):
            st = _lib.current_stream_ptr()
            _lib.check(L.vdt_q_sample(_lib.ptr(x_0), _lib.ptr(noise), _lib.ptr(coef), _lib.ptr(z_t), B, Cc * hw, st))
            out1 = teacher(z_t, t)
            z_mid, x1 = torch.empty_like(x_0), torch.empty_like(x_0)
            _lib.check(L.vdt_op_distill_step(_lib.ptr(out1), _lib.ptr(z_t), _lib.ptr(z_mid), _lib.ptr(x1), _lib.ptr(coef), B, Cc, hw,
                                             int(use_cfg), out_type, w, st))
            out2 = teacher(z_mid, t_mid)
            x_tgt, eps_tgt = torch.empty_like(x_0), torch.empty_like(x_0)
            _lib.check(L.vdt_op_distill_target(_lib.ptr(out2), _lib.ptr(z_mid), _lib.ptr(x1), _lib.ptr(z_t), _lib.ptr(x_tgt),
                                               _lib.ptr(eps_tgt), _lib.ptr(coef), B, Cc, hw, int(use_cfg), out_type, w, st))
        model_out = student_fn(z_t, t, y).to(torch.float32).contiguous()
        if tuple(model_out.shape) != (B, Cm) + tuple(x_0.shape[2:]):
            raise ValueError(f"student output has shape {tuple(model_out.shape)}, expected {(B, Cm) + tuple(x_0.shape[2:])}")
        loss = torch.empty((B,), dtype=torch.float32, device=dev)
        grad = torch.empty_like(model_out) if return_grad else None
        with torch.cuda.device(dev):
            _lib.check(L.vdt_train_loss(_lib.ptr(model_out), _lib.ptr(x_tgt), _lib.ptr(eps_tgt), _lib.ptr(z_t), _lib.ptr(coef),
                                        _lib.ptr(loss), _lib.ptr(grad), B, Cc, hw, out_type, _lib.REWEIGHT_TYPES[self.reweight_type],
                                        _lib.current_stream_ptr()))
        return (loss, grad) if return_grad else loss

    def _p_sample_generic(self, denoise_fn, shape, x_t, label, step_noise, sc, device, gen, use_ddim, solver=None, inp=None,
                          start_step=None):
        L = _lib.lib()
        B = shape[0]
        T = self.sample_timesteps
        k = T if start_step is None else start_step
        coefs = self.step_coefficients(use_ddim, solver)
        coefs[k - 1, 15] = 0.                                       # the trajectory's first step has no 2M history
        # DPM-Solver++(2M): the guided x0 of the previous step, read by every step whose c2k is non-zero
        hist = torch.empty_like(x_t) if solver is not None else None
        use_cfg = (self.w_guide > 0) and (label is not None)        # diffusion.py:368
        hw = shape[2] * shape[3]
        with torch.cuda.device(device):
            for ti in reversed(range(k)):
                t = torch.full((B,), (ti + 1) / T, dtype=torch.float64, device=device)
                if use_cfg:
                    xin, tin = x_t.repeat_interleave(2, dim=0), t.repeat_interleave(2)
                    yin = label.repeat_interleave(2, dim=0)
                    yin[1::2] = 0
                else:
                    xin, tin, yin = x_t, t, label
                model_out = denoise_fn(xin, tin, yin).to(torch.float32).contiguous()
                z = None
                if not use_ddim and ti > 0:
                    z = step_noise[ti] if step_noise is not None else torch.randn(shape, device=device, generator=gen)
                    z = z.contiguous()
                x_s = torch.empty_like(x_t)
                if inp is not None:
                    known, mask, known_noise = inp
                    _lib.check(L.vdt_op_sampler_step_known(
                        _lib.ptr(model_out), _lib.ptr(x_t), _lib.ptr(z), _lib.ptr(x_s), B, shape[1], hw, int(use_cfg),
                        sc.model_out_type, ti, _lib.ptr(coefs[ti].contiguous()), float(self.w_guide), _lib.ptr(hist),
                        _lib.ptr(known), _lib.ptr(mask), None if known_noise is None else _lib.ptr(known_noise[ti]), sc.seed,
                        _lib.ptr(coefs[ti - 1].contiguous()) if ti > 0 else None, _lib.current_stream_ptr()))
                elif hist is None:
                    _lib.check(L.vdt_op_sampler_step(_lib.ptr(model_out), _lib.ptr(x_t), _lib.ptr(z), _lib.ptr(x_s), B,
                                                     shape[1], hw, int(use_cfg), sc.model_out_type, ti,
                                                     _lib.ptr(coefs[ti].contiguous()), float(self.w_guide),
                                                     _lib.current_stream_ptr()))
                else:
                    _lib.check(L.vdt_op_sampler_step_hist(_lib.ptr(model_out), _lib.ptr(x_t), _lib.ptr(z), _lib.ptr(x_s), B,
                                                          shape[1], hw, int(use_cfg), sc.model_out_type, ti,
                                                          _lib.ptr(coefs[ti].contiguous()), float(self.w_guide), _lib.ptr(hist),
                                                          _lib.current_stream_ptr()))
                x_t = x_s
        return x_t
