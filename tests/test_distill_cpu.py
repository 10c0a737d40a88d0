"""CPU: progressive distillation's math and coefficient table (include/vdt_b200.h vdt_distill_coefficients).  The literal
Algorithm 2 of Salimans & Ho (2022) in fp64 (tests/distill_ref.py) against the closed form c_a x1 + c_b x2 the library uses,
the table against the fp64 values, and the refusals.  The host table needs no device."""
import ctypes as C

import numpy as np
import pytest
import torch

from tests import distill_ref as ref

SCHEDULES = ["cosine", "linear", "sigmoid", "legacy"]


def _steps(N):
    return sorted({0, 1, N // 2, N - 1} & set(range(N)))


@pytest.mark.parametrize("schedule", SCHEDULES)
@pytest.mark.parametrize("N", [1, 2, 7, 512])
def test_algorithm2_target_is_the_closed_form(schedule, N):
    """Two teacher DDIM steps and the paper's target formula give x~ = c_a x1 + c_b x2 (z_t cancels) to fp64 rounding, over
    random predictions; one student DDIM step from z_t with x0 = x~ lands on the teacher's z_t''."""
    g = np.random.default_rng(N * 31 + SCHEDULES.index(schedule))
    for i in _steps(N):
        lt, ltp, ltpp = ref.logsnrs(N, i, schedule)
        ca, cb = ref.closed_form(lt, ltp, ltpp)
        assert 0.0 <= ca <= 1.0 and 0.0 <= cb <= 1.0 and abs(ca + cb - 1.0) <= 1e-14, (i, ca, cb)
        z = g.standard_normal(64)
        x1 = np.clip(g.standard_normal(64), -1, 1)
        x2 = np.clip(g.standard_normal(64), -1, 1)
        _, _, z_tpp = ref.two_teacher_steps(z, x1, lambda zz: x2, lt, ltp, ltpp)
        x_lit = ref.algorithm2_target(z, z_tpp, lt, ltpp)
        x_cf = ca * x1 + cb * x2
        # the literal formula divides (z_t'' - r z_t) by alpha_t'' (1 - e^((l_t - l_t'')/2)); its own fp64 rounding is the
        # cancellation in the numerator, |z| eps64 over the denominator
        a2, s2 = ref.alpha_sigma(ltpp)
        a, s = ref.alpha_sigma(lt)
        cond = 1.0 + (np.abs(z) + np.abs(z_tpp)).max() / abs(a2 - s2 / s * a)
        err = np.abs(x_lit - x_cf).max()
        assert err <= 1e-12 * cond, (schedule, N, i, err, cond)
        # the student's step t -> t'' with x~ reproduces z_t''
        z_student = ref.ddim_step(z, x_cf, lt, ltpp)
        assert np.abs(z_student - z_tpp).max() <= 1e-12 * (1.0 + np.abs(z).max()), (schedule, N, i)


def _diffusion(N, out="v", schedule="cosine", x0eps=False):
    from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule
    return GaussianDiffusion(get_logsnr_schedule(schedule, -20., 20.), N, out, "fixed_large", "snr_trunc", "mse", x0eps_coef=x0eps)


def _train_rows(d, t):
    from v_diffusion_b200 import _lib
    sc = d.sampler_config(use_ddim=True)
    th = torch.tensor(t, dtype=torch.float64)
    out = torch.empty((len(t), _lib.COEF_STRIDE), dtype=torch.float32)
    _lib.check(_lib.lib().vdt_train_coefficients(C.byref(sc), _lib.ptr(th), len(t), _lib.ptr(out)))
    return out


@pytest.mark.parametrize("schedule", SCHEDULES)
@pytest.mark.parametrize("N", [1, 2, 7, 512])
def test_coefficient_table(schedule, N):
    """Plane 0 is vdt_train_coefficients at t bit for bit apart from slots 6-7; plane 1 the same at t'.  Slots 6-7 are the DDIM
    c1, c2 (bit-identical to the sampler's own table at 2N), 8-9 c_a, c_b, all within fp32 rounding of the fp64 values; the
    t'' = 0 rows hold (c1, c2, c_a, c_b) = (0, 1, 0, 1)."""
    d = _diffusion(N, schedule=schedule)
    steps = list(range(N)) if N <= 8 else [0, 1, 2, 100, 255, 256, 510, N - 1]
    tab = d.distill_coefficients(torch.tensor(steps))
    assert tab.shape == (2, len(steps), 16)
    t0 = _train_rows(d, [ref.times(N, i)[0] for i in steps])
    t1 = _train_rows(d, [ref.times(N, i)[1] for i in steps])
    keep0 = [k for k in range(16) if k not in (6, 7)]
    keep1 = [k for k in range(16) if k not in (6, 7, 8, 9, 10)]
    assert torch.equal(tab[0][:, keep0], t0[:, keep0])
    assert torch.equal(tab[1][:, keep1], t1[:, keep1])
    sampler = _diffusion(2 * N, schedule=schedule).step_coefficients(True)
    for r, i in enumerate(steps):
        lt, ltp, ltpp = ref.logsnrs(N, i, schedule)
        assert abs(tab[1, r, 10].item() - ltpp) <= 1e-6 * max(1.0, abs(ltpp))      # the C and numpy schedules agree to rounding
        assert torch.equal(tab[0, r, 6:8], sampler[2 * i + 1, 6:8])
        c1, c2 = ref.ddim_c1_c2(lt, ltp)
        assert np.isclose(tab[0, r, 6].item(), c1, rtol=2e-7, atol=0) and np.isclose(tab[0, r, 7].item(), c2, rtol=2e-7, atol=1e-30)
        if i == 0:
            assert tab[1, r, 6:10].tolist() == [0.0, 1.0, 0.0, 1.0]
            continue
        assert torch.equal(tab[1, r, 6:8], sampler[2 * i, 6:8])
        c1, c2 = ref.ddim_c1_c2(ltp, ltpp)
        assert np.isclose(tab[1, r, 6].item(), c1, rtol=2e-7, atol=0) and np.isclose(tab[1, r, 7].item(), c2, rtol=2e-7, atol=1e-30)
        ca, cb = ref.closed_form(lt, ltp, ltpp)
        assert abs(tab[1, r, 8].item() - ca) <= 6e-8 * ca + 1e-45 and abs(tab[1, r, 9].item() - cb) <= 6e-8 * cb + 1e-45, (i, ca, cb)
        assert tab[1, r, 8].item() >= 0 and tab[1, r, 9].item() >= 0


def _refused(d, steps, x0eps=None, N=None):
    from v_diffusion_b200 import _lib
    sc = d.sampler_config(use_ddim=True)
    if x0eps is not None:
        sc.x0eps_coef = x0eps
    if N is not None:
        sc.sample_timesteps = N
    sh = torch.tensor(steps, dtype=torch.int32)
    out = torch.empty((2, len(steps), 16), dtype=torch.float32)
    assert _lib.lib().vdt_distill_coefficients(C.byref(sc), _lib.ptr(sh), len(steps), _lib.ptr(out)) != 0
    return _lib.lib().vdt_last_error().decode()


def test_refusals():
    from v_diffusion_b200 import _lib
    d = _diffusion(4)
    assert "x0eps_coef" in _refused(d, [0], x0eps=1)
    assert ">= 1" in _refused(d, [0], N=0)
    assert "outside [0, 4)" in _refused(d, [0, 4])
    assert "outside [0, 4)" in _refused(d, [-1])
    assert _lib.lib().vdt_distill_coefficients(None, None, 0, None) != 0 and "null" in _lib.lib().vdt_last_error().decode()
    with pytest.raises(RuntimeError, match="outside"):
        d.distill_coefficients(torch.tensor([5]))
    # the kernels check their arguments before any device work
    L = _lib.lib()
    buf = torch.zeros(64)
    assert L.vdt_op_distill_step(_lib.ptr(buf), _lib.ptr(buf), _lib.ptr(buf), _lib.ptr(buf), _lib.ptr(buf), 1, 1, 4, 0, 5, 0.,
                                 None) != 0 and "unknown model_out_type 5" in L.vdt_last_error().decode()
    assert L.vdt_op_distill_target(_lib.ptr(buf), None, _lib.ptr(buf), _lib.ptr(buf), _lib.ptr(buf), _lib.ptr(buf), _lib.ptr(buf),
                                   1, 1, 4, 0, 3, 0., None) != 0 and "null" in L.vdt_last_error().decode()
    assert L.vdt_op_distill_step(_lib.ptr(buf), _lib.ptr(buf), _lib.ptr(buf), _lib.ptr(buf), _lib.ptr(buf), 1, 0, 4, 0, 3, 0.,
                                 None) != 0 and "bad image shape" in L.vdt_last_error().decode()


def test_python_refusals():
    d = _diffusion(4)
    with pytest.raises(RuntimeError, match="CUDA"):
        d.distill_loss(lambda *a: None, lambda *a: None, torch.zeros(2, 3, 4, 4), torch.tensor([0, 1]), None)


@pytest.mark.parametrize("argv,msg", [(["--teacher-steps", "6", "--stages", "2"], "multiple of 2^stages"),
                                      (["--teacher-steps", "8", "--iters", "0"], ">= 1"),
                                      (["--teacher-steps", "8", "--w-guide", "-1"], "--w-guide")])
def test_driver_refuses_bad_arguments(argv, msg, capsys):
    from v_diffusion_b200 import distill
    base = ["--config-path", "c.json", "--ckpt-path", "c.pt", "--images", "x.npy", "--out-dir", "o"]
    if "--iters" not in argv:
        base += ["--iters", "1"]
    with pytest.raises(SystemExit):
        distill.main(base + argv)
    assert msg in capsys.readouterr().err
