"""Child process of tests/test_train_mnist28_gpu.py: one whole-network training case at 28x28 on cuda:0 (wgrad on tiles of 112 and
98 pixels).  Prints one JSON line.

    python -m tests.mnist28_train_worker graph_parity mnist_cfg3 2 fp16
    python -m tests.mnist28_train_worker graph_parity mnist28 3 bf16
    python -m tests.mnist28_train_worker train_steps mnist_cfg3 2 fp16
    python -m tests.mnist28_train_worker train_then_sample mnist_cfg3 2 fp16
"""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tests import train_step_worker as tsw                               # noqa: E402
from tests.cases import _cfg, UNET_CASES                                 # noqa: E402
from v_diffusion_b200 import UNet, GaussianDiffusion, get_logsnr_schedule   # noqa: E402
from v_diffusion_b200.training import TrainingStep                       # noqa: E402

CASES = {
    # BASELINE configs[3]'s network: the defaults model block with 1 input / output channel, hid 256, mult 1-1-1, 3 residual
    # blocks, attention at 14x14 and 7x7 (and in the upsampling block to 28x28), 10 classes; 414 tensors, 60.8 M parameters
    "mnist_cfg3": dict(cfg=_cfg(in_channels=1, hid=256, out_channels=1, mult=(1, 1, 1), nrb=3, attn=(False, True, True),
                                num_classes=10), res=28),
    # hid 64, mult 1-2-2: 2-channel groups, wgrad cout 64 (a lone 64-channel block) and 128 on ragged tiles; 236 tensors
    "mnist28": dict(cfg=UNET_CASES["mnist28"]["cfg"], res=28),
}
tsw.CASES.update(CASES)                                                   # graph_parity / train_steps look their case up there


def train_then_sample(case, B, operand, steps=3):
    """The user's loop at 28x28: sample once (this builds the 28x28 sampling plan from the initial weights), take three
    TrainingStep.step's with configs[3]'s objective, then TrainingStep.sample_fn -- CFG w = 3 ancestral with the EMA weights.
    That sample must equal, bit for bit, p_sample on the same seed from a fresh UNet loaded with the EMA shadow: the re-pack
    after the steps (mark_weights_changed) reached the plan."""
    cfg, R = CASES[case]["cfg"], CASES[case]["res"]
    sd, net = tsw.build(cfg, 37, operand)
    net.train()
    diff = GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), 100, "v", "fixed_medium", "snr_trunc", "mse",
                             intp_frac=0.3, w_guide=3.0, p_uncond=0.1)          # w_guide only matters to sampling
    ts = TrainingStep(net, diff, timesteps=0, lr=2e-4, weight_decay=0.001, grad_norm=1.0, use_ema=True, ema_decay=0.9999)
    shape, label, seed = (B, cfg["in_channels"], R, R), torch.arange(B) % cfg["num_classes"] + 1, 4242
    before = ts.sample_fn(shape, label=label, use_ddim=False, seed=seed)
    g = torch.Generator().manual_seed(79)
    losses = []
    for _ in range(steps):
        x = torch.randn(B, cfg["in_channels"], R, R, generator=g).clamp(-1, 1)
        y = torch.randint(1, cfg["num_classes"] + 1, (B,), generator=g)
        losses.append(float(ts.step(x.cuda(), y.cuda())))
    after = ts.sample_fn(shape, label=label, use_ddim=False, seed=seed)
    fresh = UNet(cfg["in_channels"], cfg["hid_channels"], cfg["out_channels"], cfg["ch_multipliers"], cfg["num_res_blocks"],
                 cfg["apply_attn"], embedding_dim=cfg["embedding_dim"], head_dim=cfg["head_dim"], num_heads=cfg["num_heads"],
                 num_classes=cfg["num_classes"], multitags=cfg["multitags"])
    fresh.load_state_dict({k: v.detach().cpu() for k, v in ts.optimizer.shadow.items()}, strict=True)
    fresh.operand_dtype = operand
    fresh = fresh.cuda().eval()
    ref = diff.p_sample(fresh, shape, device="cuda", label=label.cuda(), seed=seed, use_ddim=False)
    return dict(bit_identical=bool(torch.equal(after, ref)), max_abs_diff=float((after - ref).abs().max()),
                moved_by_training=float((after - before).abs().max()), finite=bool(torch.isfinite(after).all()),
                sample_abs_max=float(after.abs().max()), losses=losses)


if __name__ == "__main__":
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.cuda.set_device(0)
    kind, case, B, operand = sys.argv[1], sys.argv[2], int(sys.argv[3]), sys.argv[4]
    res = {"graph_parity": tsw.graph_parity, "train_steps": tsw.train_steps, "train_then_sample": train_then_sample}[kind](case, B, operand)
    print("RESULT " + json.dumps(res))
