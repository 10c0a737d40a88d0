"""Child process of tests/test_train_step_gpu.py: runs one case of the composed training step on cuda:0 and prints one JSON
line.  (A child, so that a device fault in this newest code path cannot take the rest of the GPU suite with it.)

    python -m tests.train_step_worker graph_parity cifar_cond 4 fp16
    python -m tests.train_step_worker train_steps small 8 fp16
    python -m tests.train_step_worker dropout small 4 fp16
    python -m tests.train_step_worker grad_golden cifar 0 fp16
"""
import json
import math
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import make_state_dict, train_loss as oracle_train_loss      # noqa: E402
from oracle.unet_ref import _unet_forward                                # noqa: E402
from tests.cases import _cfg, CIFAR_COND                                 # noqa: E402
from v_diffusion_b200 import UNet, GaussianDiffusion, get_logsnr_schedule, _lib   # noqa: E402
from v_diffusion_b200.training import UNetTrainGraph, TrainingStep       # noqa: E402

CASES = {
    # BASELINE configs[4]'s network: cifar10_cond.json (hid 256, three levels, attention at 16x16 and 8x8, 10 classes)
    "cifar_cond": dict(cfg=CIFAR_COND, res=32),
    # every block type at a quarter of the cost: 128 / 256-channel norms, 1x1 skips, avg-pool + upsample blocks, one attention level
    "small": dict(cfg=_cfg(hid=128, mult=(1, 1), nrb=1, attn=(False, True), num_classes=10), res=16),
}


def build(cfg, seed, operand, drop_rate=0.0):
    sd = make_state_dict(cfg, seed)
    net = UNet(cfg["in_channels"], cfg["hid_channels"], cfg["out_channels"], cfg["ch_multipliers"], cfg["num_res_blocks"],
               cfg["apply_attn"], embedding_dim=cfg["embedding_dim"], drop_rate=drop_rate, head_dim=cfg["head_dim"],
               num_heads=cfg["num_heads"], num_classes=cfg["num_classes"], multitags=cfg["multitags"])
    net.load_state_dict(sd, strict=True)
    net.operand_dtype = operand
    return sd, net.cuda()


def rel(a, b, floor=0.0):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return ((a - b).norm() / (b.norm() + floor)).item()


def inputs(cfg, B, R, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, cfg["in_channels"], R, R, generator=g)
    t = torch.rand(B, generator=g, dtype=torch.float64)
    go = torch.randn(B, cfg["out_channels"], R, R, generator=g)
    y = torch.randint(0, cfg["num_classes"] + 1, (B,), generator=g) if cfg["num_classes"] else None
    if y is not None:
        y[0] = 0                                                           # one unconditional row
    return x, t, y, go


def graph_parity(case, B, operand):
    """UNetTrainGraph forward + backward on the kernels vs fp32 autograd through the oracle UNet on the CPU."""
    cfg, R = CASES[case]["cfg"], CASES[case]["res"]
    sd, net = build(cfg, 17, operand)
    x, t, y, go = inputs(cfg, B, R, 5)
    n0 = _lib.lib().vdt_kernel_launches()
    graph = UNetTrainGraph(net)
    out = graph.forward(x.cuda(), t.cuda(), None if y is None else y.cuda())
    grads = graph.backward(go.cuda() * 1e-4)                               # small like d loss.mean() / d out: exercises the fp16 scaling
    torch.cuda.synchronize()
    launches = int(_lib.lib().vdt_kernel_launches() - n0)
    ref_sd = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    with torch.enable_grad():
        ref = _unet_forward(ref_sd, cfg, x, t, y, None)
        ref.backward(go * 1e-4)
    errs = {}
    for k in sd:
        want = ref_sd[k].grad
        errs[k] = rel(grads[k], want, floor=1e-3 * 1e-4 * math.sqrt(want.numel()))
    worst = sorted(errs.items(), key=lambda kv: -kv[1])[:5]
    finite = all(bool(torch.isfinite(g).all()) for g in grads.values())
    return dict(out_rel=rel(out, ref), grad_rel_worst=worst[0][1], worst=worst, finite=finite, launches=launches,
                n_params=len(sd), grad_rel_median=sorted(errs.values())[len(errs) // 2])


def train_steps(case, B, operand, steps=3):
    """TrainingStep.step (draws, q_sample, forward, loss, backward, clip, AdamW, EMA) for a few steps vs the same steps done
    with the oracle UNet under autograd + torch.optim.AdamW + clip_grad_norm_ + the reference's EMA formula on the CPU, fed
    the very same (t, noise) draws."""
    cfg, R = CASES[case]["cfg"], CASES[case]["res"]
    sd, net = build(cfg, 23, operand)
    net.train()                                                            # drop_rate 0: .train() changes nothing else
    diff = GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), 100, "v", "fixed_medium", "snr_trunc", "mse",
                             intp_frac=0.3, p_uncond=0.1)
    lr, wd, gn, decay = 2e-4, 0.001, 1.0, 0.9999
    ts = TrainingStep(net, diff, timesteps=0, lr=lr, weight_decay=wd, grad_norm=gn, use_ema=True, ema_decay=decay)
    ref_p = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    opt = torch.optim.AdamW(list(ref_p.values()), lr=lr, weight_decay=wd)
    shadow = {k: v.detach().clone() for k, v in ref_p.items()}
    twin = torch.Generator("cuda").manual_seed(8191)                       # replays TrainingStep.draw's stream
    g = torch.Generator().manual_seed(77)
    rec = dict(loss=[], loss_ref=[], gnorm=[], gnorm_ref=[])
    for s in range(steps):
        x = torch.randn(B, cfg["in_channels"], R, R, generator=g).clamp(-1, 1)
        y = torch.randint(1, cfg["num_classes"] + 1, (B,), generator=g)
        t = torch.rand((B,), dtype=torch.float64, device="cuda", generator=twin)
        noise = torch.empty(x.shape, device="cuda").normal_(generator=twin)
        loss = ts.step(x.cuda(), y.cuda())
        rec["loss"].append(float(loss))
        rec["gnorm"].append(math.sqrt(float(ts.last_grad_sq)))
        with torch.enable_grad():
            per, _ = oracle_train_loss(lambda a, b, c: _unet_forward(ref_p, cfg, a, b, c, None), x, t.cpu(), y, noise.cpu(),
                                       model_out_type="v", reweight_type="snr_trunc")
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
    ema = max(rel(ts.optimizer.shadow[k], shadow[k]) for k in shadow)
    return dict(cosine_of_updates=cos, update_norm_ratio=float(upd.norm() / upd_ref.norm()), ema_rel_worst=ema,
                loss_rel_worst=max(abs(a - b) / abs(b) for a, b in zip(rec["loss"], rec["loss_ref"])),
                gnorm_rel_worst=max(abs(a - b) / abs(b) for a, b in zip(rec["gnorm"], rec["gnorm_ref"])), **rec)


def dropout(case, B, operand):
    """.train() with drop_rate 0.2 (cifar10_cond.json): the step is reproducible for a fixed seed, differs across seeds and from
    .eval(); the masks drop ~20 %; out_conv's bias gradient (independent of any mask) still equals sum(go)."""
    cfg, R = CASES[case]["cfg"], CASES[case]["res"]
    sd, net = build(cfg, 29, operand, drop_rate=0.2)
    net.train()
    x, t, y, go = inputs(cfg, B, R, 9)
    graph = UNetTrainGraph(net)
    xs, tc, yc, goc = x.cuda(), t.cuda(), y.cuda(), go.cuda()
    a = graph.forward(xs, tc, yc, seed=42); ga = graph.backward(goc)
    b = graph.forward(xs, tc, yc, seed=42); gb = graph.backward(goc)
    c = graph.forward(xs, tc, yc, seed=43); graph.backward(goc)
    net.eval()
    e = graph.forward(xs, tc, yc); graph.backward(goc)
    same = bool(torch.equal(a, b)) and all(bool(torch.equal(ga[k], gb[k])) for k in ga)
    finite = all(bool(torch.isfinite(v).all()) for v in ga.values())
    bias_rel = rel(ga["out_conv.2.bias"], go.sum(dim=(0, 2, 3)))
    return dict(reproducible=same, finite=finite, seed_changes_output=rel(c, a), eval_differs=rel(e, a), out_bias_grad_rel=bias_rel)


def vs_grad_fixture(case, loss, grads):
    """Per-sample loss and parameter gradients against tests/golden/train_grads_<case>.npz, made by the UNMODIFIED reference's own
    UNet / train_loss / autograd (tests/golden/make_train_grad_golden.py): every gradient's norm and probe projection, the small
    tensors in full."""
    import numpy as np
    from tests.cases import grad_probe
    g = np.load(os.path.join(ROOT, "tests", "golden", f"train_grads_{case}.npz"))
    loss_rel = float(np.abs(loss.detach().cpu().numpy() - g["loss"]).max() / np.abs(g["loss"]).max())
    norm_err, proj_err, full_err = {}, {}, {}
    for k in (str(n) for n in g["names"]):
        gr = grads[k].detach().double().cpu()
        n_ref = float(g["norm/" + k])
        norm_err[k] = abs(gr.norm().item() - n_ref) / n_ref
        proj_err[k] = abs((gr * grad_probe(k, gr.shape)).sum().item() - float(g["proj/" + k])) / n_ref
        if ("full/" + k) in g.files:
            full_err[k] = (gr - torch.from_numpy(g["full/" + k]).double()).norm().item() / n_ref
    top = lambda d: sorted(d.items(), key=lambda kv: -kv[1])[:3]
    return dict(loss_rel=loss_rel, norm_rel_worst=top(norm_err)[0][1], proj_err_worst=top(proj_err)[0][1],
                full_rel_worst=top(full_err)[0][1], n_params=len(norm_err), n_full=len(full_err),
                worst=dict(norm=top(norm_err), proj=top(proj_err), full=top(full_err)))


def grad_golden(case, B, operand):
    """TrainingStep.loss_and_grads on the kernels against the reference's gradient fixture (vs_grad_fixture).  (B comes from the
    fixture.)"""
    from tests.cases import TRAIN_GRAD_CASES, build_train_grad_inputs
    c = TRAIN_GRAD_CASES[case]                                         # "small" | "cifar" (cifar10_cond.json's own network)
    sd, net = build(c["cfg"], c["wseed"], operand)
    net.train()
    diff = GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), 1000, c["model_out_type"], "fixed_medium", c["reweight_type"],
                             "mse", intp_frac=0.3, p_uncond=0.1)
    ts = TrainingStep(net, diff, timesteps=0)
    x0, t, noise, y = build_train_grad_inputs(c)
    loss, grads = ts.loss_and_grads(x0.cuda(), y.cuda(), t=t.cuda(), noise=noise.cuda())
    torch.cuda.synchronize()
    return vs_grad_fixture(case, loss, grads)


def autograd_step(case, B, operand):
    """UNet.autograd = True on the GPU as the denoise_fn of train_loss (the oracle's restatement, pinned to the reference's), then
    loss.mean().backward() as in Trainer.step (train_utils.py:149-151): loss and every parameter's .grad against the reference's
    gradient fixture (vs_grad_fixture).  (B comes from the fixture.)"""
    from tests.cases import TRAIN_GRAD_CASES, build_train_grad_inputs
    c = TRAIN_GRAD_CASES[case]
    sd, net = build(c["cfg"], c["wseed"], operand)
    net.autograd = True
    net.train()
    x0, t, noise, y = build_train_grad_inputs(c)
    with torch.enable_grad():
        loss, _ = oracle_train_loss(lambda a, b, yy: net(a.cuda(), b.cuda(), yy.cuda()).cpu(), x0, t, y.clone(), noise,
                                    model_out_type=c["model_out_type"], reweight_type=c["reweight_type"])
        loss.mean().backward()
    torch.cuda.synchronize()
    res = vs_grad_fixture(case, loss, {k: p.grad for k, p in net.named_parameters()})
    with torch.no_grad():
        sampled = net(x0.cuda(), t.cuda(), y.cuda())                       # no grad mode: still the plan path (dropout 0 here)
    return dict(res, plan_path_finite=bool(torch.isfinite(sampled).all()))


if __name__ == "__main__":
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.cuda.set_device(0)
    kind, case, B, operand = sys.argv[1], sys.argv[2], int(sys.argv[3]), sys.argv[4]
    res = {"graph_parity": graph_parity, "train_steps": train_steps, "dropout": dropout, "autograd_step": autograd_step,
           "grad_golden": grad_golden}[kind](case, B, operand)
    print("RESULT " + json.dumps(res))
