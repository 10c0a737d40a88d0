"""GPU: progressive distillation (include/vdt_b200.h vdt_distill_coefficients; GaussianDiffusion.distill_loss, DistillationStep,
python -m v_diffusion_b200.distill).  Each case runs in a child process (tests/distill_worker.py).  Bars on measured values sit
2-5x above what a B200 measured (profiles/r11_distill_parity.txt)."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, timeout=900):
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run([sys.executable, "-m", "tests.distill_worker", *map(str, args)], cwd=ROOT, env=env, capture_output=True,
                       text=True, timeout=timeout)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")]
    assert r.returncode == 0 and lines, (r.stdout[-1500:] + "\n" + r.stderr[-2500:])
    res = json.loads(lines[-1][len("RESULT "):])
    print(" ".join(map(str, args)), "->", json.dumps(res)[:3000])
    return res


def test_kernels_vs_fp64():
    """distill_step_kernel and distill_target_kernel against the fp64 restatement from the same fp32 rows, for the four out
    types x CFG off / on x {aligned, offset by one float, odd C*H*W}: errors in units of the terms' magnitudes stay at fp32
    rounding, as test_inversion_gpu.py bounds the inversion kernel."""
    res = _run("kernels")
    assert len(res["cases"]) == 24
    assert res["worst"] <= 1e-6, res


def test_closed_form_loss_and_gradient_vanish():
    """Gaussian data with the analytic denoiser as teacher and a student that returns the exact analytic target: the distillation
    loss and its gradient are zero up to fp32 noise (measured 1.4e-14 and 7.5e-10 for v and x0), with w_guide 0 and 1 and v, x0
    and eps outputs."""
    res = _run("closed_form")
    assert res["loss_worst"] <= 1e-12 and res["grad_worst"] <= 1e-8, res


@pytest.mark.parametrize("w", [0.0, 1.0])
def test_distillation_step_vs_autograd(w):
    """One DistillationStep against the oracle UNet under fp32 autograd on the same draws (B = 4, a small conditional network as
    teacher and student, drop_rate 0): the loss and every student gradient within the training step's bars (8e-3 rel-L2 with
    fp16 operands); three optimizer steps follow AdamW + EMA as in test_training_steps_follow_the_reference_recipe."""
    res = _run("composed", w)
    assert res["grad_rel_worst"] <= 8e-3, res["worst"]
    assert res["loss_rel_worst"] <= 1e-3 and res["gnorm_rel_worst"] <= 1e-3, res
    assert res["cosine_of_updates"] >= 0.999 and 0.999 <= res["update_norm_ratio"] <= 1.001, res
    assert res["ema_rel_worst"] <= 3e-3, res


def test_distillation_halves_the_step_gap():
    """An unconditional hid-64 network at 16^2, trained for 400 steps on synthetic data, distilled from 8 to 4 DDIM steps in 600
    iterations: the student's 4-step samples are at most half as far (RMS) from the teacher's 8-step samples as the teacher's
    own 4-step samples, and the loss falls.  (A random-weight teacher is no denoiser: its 4- and 8-step samples differ little,
    and the student fell short of them; measured ratios in profiles/r11_distill_parity.txt.)"""
    res = _run("works", timeout=600)
    assert res["finite"], res
    assert res["ratio"] <= 0.5, res
    assert res["loss_last"] < res["loss_first"], res


def test_driver_round_trip():
    res = _run("driver")
    assert res["stages_seen"] == 2 and res["stage1_teacher_is_ckpt"], res
    assert res["stage2_teacher_is_stage1_ema"] and res["ema_differs_from_teacher"], res
    assert res["keys"] == dict(sample_timesteps=4, distill_w_guide=0.0, has_optimizer=True, has_ema=True), res
    assert res["student_2_exists"] and res["sample_finite"] and res["sample_shape"] == [4, 3, 32, 32], res
