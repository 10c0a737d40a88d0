"""Child process of tests/test_train_celeba_gpu.py: one whole-network training case on cuda:0 for the networks whose widths need
the generalised backward kernels (GroupNorm backward at any C % 64 == 0, wgrad at cout % 128 == 64).  Prints one JSON line.

    python -m tests.celeba_train_worker graph_parity celeba 2 fp16
    python -m tests.celeba_train_worker graph_parity narrow 3 bf16
    python -m tests.celeba_train_worker train_steps celeba_multitag 2 fp16
"""
import json
import math
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import train_loss as oracle_train_loss                       # noqa: E402
from oracle.unet_ref import _unet_forward                                # noqa: E402
from tests import train_step_worker as tsw                               # noqa: E402
from tests.cases import CELEBA, UNET_CASES                               # noqa: E402
from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule      # noqa: E402
from v_diffusion_b200.training import TrainingStep                       # noqa: E402

CASES = {
    # celeba.json's network: hid 192, mult 1-2-3-4, E 768, 64-wide heads, 6 output channels ("both"), 64x64 -> 8x8.  GroupNorm
    # widths 192 / 384 / 576 / 768 and concat widths 960 / 1152 / 1344 / 1536; wgrad cout 192 and 576 (64-channel tail block)
    "celeba": dict(cfg=CELEBA, res=64),
    # the same with celeba.json's 40-way multitag conditioning (the reference's conditional CelebA checkpoints)
    "celeba_multitag": dict(cfg=dict(CELEBA, num_classes=40, multitags=True), res=64),
    # hid 64: 2- and 6-channel groups (64, 192), concat widths 128 / 192 / 256, wgrad cout 64 (a lone tail block)
    "narrow": dict(cfg=UNET_CASES["small_cond"]["cfg"], res=16),
}
tsw.CASES.update(CASES)                                                   # graph_parity looks its case up there


def graph_parity(case, B, operand):
    """UNetTrainGraph forward + backward on the kernels vs fp32 autograd through the oracle UNet (tests/train_step_worker.py)."""
    return tsw.graph_parity(case, B, operand)


def train_steps(case, B, operand, steps=3):
    """Three TrainingStep.step's with celeba.json's objective -- "both" output, fixed_large, snr_trunc, intp_frac 0, p_uncond 0.1,
    multitag labels -- vs the same steps with the oracle UNet under autograd + clip_grad_norm_ + torch.optim.AdamW + the
    reference's EMA on the CPU, fed the very same (t, noise) draws.  drop_rate 0: the oracle cannot replay the kernels' mask."""
    cfg, R = CASES[case]["cfg"], CASES[case]["res"]
    sd, net = tsw.build(cfg, 31, operand)
    net.train()
    diff = GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), 256, "both", "fixed_large", "snr_trunc", "mse",
                             intp_frac=0.0, p_uncond=0.1)
    lr, wd, gn, decay = 2e-4, 0.001, 1.0, 0.9999
    ts = TrainingStep(net, diff, timesteps=0, lr=lr, weight_decay=wd, grad_norm=gn, use_ema=True, ema_decay=decay)
    ref_p = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    opt = torch.optim.AdamW(list(ref_p.values()), lr=lr, weight_decay=wd)
    shadow = {k: v.detach().clone() for k, v in ref_p.items()}
    twin = torch.Generator("cuda").manual_seed(8191)                       # replays TrainingStep.draw's stream
    g = torch.Generator().manual_seed(78)
    rec = dict(loss=[], loss_ref=[], gnorm=[], gnorm_ref=[])
    for s in range(steps):
        x = torch.randn(B, cfg["in_channels"], R, R, generator=g).clamp(-1, 1)
        y = (torch.rand(B, cfg["num_classes"], generator=g) < 0.12).float()   # ~5 of 40 attributes per image
        y[0] = 0                                                               # one row without attributes
        t = torch.rand((B,), dtype=torch.float64, device="cuda", generator=twin)
        noise = torch.empty(x.shape, device="cuda").normal_(generator=twin)
        loss = ts.step(x.cuda(), y.cuda())
        rec["loss"].append(float(loss))
        rec["gnorm"].append(math.sqrt(float(ts.last_grad_sq)))
        with torch.enable_grad():
            per, _ = oracle_train_loss(lambda a, b, c: _unet_forward(ref_p, cfg, a, b, c, None), x, t.cpu(), y, noise.cpu(),
                                       model_out_type="both", reweight_type="snr_trunc")
            opt.zero_grad(set_to_none=True)
            per.mean().backward()
        rec["loss_ref"].append(float(per.mean().detach()))
        rec["gnorm_ref"].append(float(torch.nn.utils.clip_grad_norm_(list(ref_p.values()), max_norm=gn)))
        opt.step()
        d = min(decay, (1 + s + 1) / (10 + s + 1))
        with torch.no_grad():
            for k in shadow:
                shadow[k] += (1 - d) * (ref_p[k] - shadow[k])
    torch.cuda.synchronize()
    upd, upd_ref = [], []
    for k, p in net.named_parameters():
        upd.append((p.detach().cpu() - sd[k]).reshape(-1))
        upd_ref.append((ref_p[k].detach() - sd[k]).reshape(-1))
    upd, upd_ref = torch.cat(upd).double(), torch.cat(upd_ref).double()
    cos = float((upd @ upd_ref) / (upd.norm() * upd_ref.norm()))
    ema = max(tsw.rel(ts.optimizer.shadow[k], shadow[k]) for k in shadow)
    return dict(cosine_of_updates=cos, update_norm_ratio=float(upd.norm() / upd_ref.norm()), ema_rel_worst=ema, n_params=len(sd),
                loss_rel_worst=max(abs(a - b) / abs(b) for a, b in zip(rec["loss"], rec["loss_ref"])),
                gnorm_rel_worst=max(abs(a - b) / abs(b) for a, b in zip(rec["gnorm"], rec["gnorm_ref"])), **rec)


if __name__ == "__main__":
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.cuda.set_device(0)
    kind, case, B, operand = sys.argv[1], sys.argv[2], int(sys.argv[3]), sys.argv[4]
    res = {"graph_parity": graph_parity, "train_steps": train_steps}[kind](case, B, operand)
    print("RESULT " + json.dumps(res))
