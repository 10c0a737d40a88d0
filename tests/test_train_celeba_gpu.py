"""GPU: the composed training step on the networks whose widths need the generalised backward kernels -- celeba.json's network
(GroupNorm backward at 192 ... 1536 channels, wgrad with cout 192 / 576) and a hid-64 network (2- and 6-channel groups, wgrad
cout 64).  Each case runs in a child process (tests/celeba_train_worker.py), as tests/test_train_step_gpu.py does.

The reference is fp32 autograd through the oracle UNet on the CPU; the bars are those of the CIFAR cases in
tests/test_train_step_gpu.py.  Measured values: DESIGN.md §7 and profiles/r3_celeba_train_parity.txt.
"""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
BARS = {"fp16": (3e-3, 8e-3), "bf16": (2.5e-2, 5e-2)}          # (output rel-L2, worst parameter-gradient rel-L2)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, timeout=1800):
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run([sys.executable, "-m", "tests.celeba_train_worker", *map(str, args)], cwd=ROOT, env=env, capture_output=True,
                       text=True, timeout=timeout)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")]
    assert r.returncode == 0 and lines, (r.stdout[-1500:] + "\n" + r.stderr[-2500:])
    res = json.loads(lines[-1][len("RESULT "):])
    print(" ".join(map(str, args)), "->", json.dumps(res)[:1200])
    return res


@pytest.mark.parametrize("case,B,operand", [("celeba", 2, "fp16"), ("narrow", 3, "fp16"), ("narrow", 3, "bf16")])
def test_unet_forward_backward_on_kernels_vs_autograd(case, B, operand):
    """Output and every parameter gradient of UNet forward + backward composed from the library's kernels against fp32 autograd
    through the oracle UNet; `celeba` is celeba.json's network at 64x64 (570 parameter tensors), `narrow` a hid-64 network."""
    res = _run("graph_parity", case, B, operand)
    assert res["finite"] and res["launches"] > 100
    if case == "celeba":
        assert res["n_params"] == 570, res["n_params"]
    assert res["out_rel"] <= BARS[operand][0], res
    assert res["grad_rel_worst"] <= BARS[operand][1], res["worst"]


def test_celeba_training_steps_follow_the_reference_recipe():
    """Three TrainingStep.step's of celeba.json's network and objective ("both", fixed_large, snr_trunc, intp_frac 0, p_uncond 0.1,
    40-way multitag labels) at batch 2 against oracle autograd + clip_grad_norm_ + torch.optim.AdamW + the reference EMA on the
    same draws, with the bars of test_training_steps_follow_the_reference_recipe."""
    res = _run("train_steps", "celeba_multitag", 2, "fp16")
    assert res["loss_rel_worst"] <= 1e-3, res
    assert res["gnorm_rel_worst"] <= 2e-3, res
    assert res["cosine_of_updates"] >= 0.999 and 0.999 <= res["update_norm_ratio"] <= 1.001, res
    assert res["ema_rel_worst"] <= 3e-3, res
