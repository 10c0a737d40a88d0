"""GPU: the composed training step on 28x28 networks, whose 3x3 / 1x1 weight gradients run wgrad on tiles of 112 (28x28) and 98
(14x14, 7x7) pixels -- BASELINE configs[3]'s network and the small MNIST-style one (tests.cases.UNET_CASES["mnist28"]).  Each
case runs in a child process (tests/mnist28_train_worker.py), as tests/test_train_step_gpu.py does.

The reference is fp32 autograd through the oracle UNet on the CPU; the bars are those of tests/test_train_celeba_gpu.py.
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
    r = subprocess.run([sys.executable, "-m", "tests.mnist28_train_worker", *map(str, args)], cwd=ROOT, env=env, capture_output=True,
                       text=True, timeout=timeout)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")]
    assert r.returncode == 0 and lines, (r.stdout[-1500:] + "\n" + r.stderr[-2500:])
    res = json.loads(lines[-1][len("RESULT "):])
    print(" ".join(map(str, args)), "->", json.dumps(res)[:1200])
    return res


@pytest.mark.parametrize("case,B,operand,n_params", [("mnist_cfg3", 2, "fp16", 414), ("mnist28", 3, "fp16", 236),
                                                     ("mnist28", 3, "bf16", 236)])
def test_mnist28_forward_backward_on_kernels_vs_autograd(case, B, operand, n_params):
    """Output and every parameter gradient of UNet forward + backward composed from the library's kernels against fp32 autograd
    through the oracle UNet at 28x28; `mnist_cfg3` is BASELINE configs[3]'s network, `mnist28` a hid-64 one."""
    res = _run("graph_parity", case, B, operand)
    assert res["finite"] and res["launches"] > 100
    assert res["n_params"] == n_params, res["n_params"]
    assert res["out_rel"] <= BARS[operand][0], res
    assert res["grad_rel_worst"] <= BARS[operand][1], res["worst"]


def test_mnist28_training_steps_follow_the_reference_recipe():
    """Three TrainingStep.step's of configs[3]'s network with cifar10_cond.json's objective (v, fixed_medium, snr_trunc, intp_frac
    0.3, p_uncond 0.1, class ids 1..10) at batch 2 against oracle autograd + clip_grad_norm_ + torch.optim.AdamW + the reference EMA
    on the same draws, with the bars of test_celeba_training_steps_follow_the_reference_recipe."""
    res = _run("train_steps", "mnist_cfg3", 2, "fp16")
    assert res["loss_rel_worst"] <= 1e-3, res
    assert res["gnorm_rel_worst"] <= 2e-3, res
    assert res["cosine_of_updates"] >= 0.999 and 0.999 <= res["update_norm_ratio"] <= 1.001, res
    assert res["ema_rel_worst"] <= 3e-3, res


def test_mnist28_train_then_sample_uses_the_trained_ema_weights():
    """Train configs[3]'s network for three steps, then TrainingStep.sample_fn (CFG w = 3, ancestral): bit-identical to p_sample
    from a fresh UNet loaded with the EMA shadow on the same seed, and different from the sample taken before training."""
    res = _run("train_then_sample", "mnist_cfg3", 2, "fp16")
    assert res["finite"], res
    assert res["bit_identical"], res
    assert res["moved_by_training"] > 0, res
