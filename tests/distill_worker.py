"""Child process of tests/test_distill_gpu.py: one progressive-distillation case on cuda:0.  Prints one JSON line.

    python -m tests.distill_worker kernels
    python -m tests.distill_worker closed_form
    python -m tests.distill_worker composed 1.0
    python -m tests.distill_worker works
    python -m tests.distill_worker driver
"""
import json
import math
import os
import sys
import tempfile
import zlib

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import make_state_dict, train_loss as oracle_train_loss       # noqa: E402
from oracle.diffusion_ref import logsnr_schedule                          # noqa: E402
from oracle.unet_ref import _unet_forward                                 # noqa: E402
from tests import distill_ref as ref                                      # noqa: E402
from tests.cases import _cfg                                              # noqa: E402
from v_diffusion_b200 import UNet, GaussianDiffusion, get_logsnr_schedule, _lib   # noqa: E402
from v_diffusion_b200.training import DistillationStep                   # noqa: E402

OUT_TYPES = ["x0", "eps", "both", "v"]


def _diffusion(N, out="v", reweight="snr_trunc", p_uncond=0.1):
    return GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), N, out, "fixed_large", reweight, "mse", p_uncond=p_uncond)


def _net(cfg, sd, drop_rate=0.0):
    net = UNet(cfg["in_channels"], cfg["hid_channels"], cfg["out_channels"], cfg["ch_multipliers"], cfg["num_res_blocks"],
               cfg["apply_attn"], embedding_dim=cfg["embedding_dim"], drop_rate=drop_rate, head_dim=cfg["head_dim"],
               num_heads=cfg["num_heads"], num_classes=cfg["num_classes"], multitags=cfg["multitags"])
    net.load_state_dict(sd, strict=True)
    return net.cuda()


def _offset(t, off):
    buf = torch.empty(t.numel() + off, device="cuda")
    v = buf[off:].view(t.shape)
    v.copy_(t)
    return v


def _x0_mag(x, out, cf, t):
    """|terms| of the per-branch x0 (the scale of its fp32 rounding)."""
    if t == "x0":
        return out.abs()
    if t == "v":
        return (x * cf[0]).abs() + (out * cf[1]).abs()
    if t == "eps":
        return (x * cf[2]).abs() + (out * cf[3]).abs()
    xo, eo = out.chunk(2, dim=1)
    return (xo * cf[5]).abs() + ((x * cf[2]).abs() + (eo * cf[3]).abs()) * cf[4]


def _x0_fp64(x, out, cf, t, w, cfg):
    """Guided, clipped x0 per sample from the fp32 row cf ([B, 16] fp64) and its magnitude scale."""
    c = cf.reshape(cf.shape[0], 16, 1, 1, 1).transpose(0, 1)            # slot k -> (B, 1, 1, 1)
    x = x.double()
    out = out.double()

    def one(o):
        if t == "x0":
            v = o
        elif t == "v":
            v = x * c[0] - o * c[1]
        elif t == "eps":
            v = x * c[2] - o * c[3]
        else:
            xo, eo = o.chunk(2, dim=1)
            v = xo * c[5] + (x * c[2] - eo * c[3]) * c[4]
        return v.clamp(-1., 1.), _x0_mag(x, o, c, t)
    if not cfg:
        return one(out)
    (xc, mc), (xu, mu) = one(out[0::2]), one(out[1::2])
    return xc + w * (xc - xu), (1 + w) * mc + w * mu


def kernels():
    """Both kernels against the fp64 restatement from the same fp32 rows: every out type x CFG off/on x {aligned, offset by
    one float, odd C*H*W}; errors in units of the terms' magnitude."""
    L = _lib.lib()
    N, B, Cc, w = 7, 5, 3, 1.5
    res = {}
    for t in OUT_TYPES:
        d = _diffusion(N, t)
        for cfg in (False, True):
            for hw, off in (((16, 16), 0), ((16, 16), 1), ((5, 7), 0)):
                g = torch.Generator().manual_seed(zlib.crc32(f"{t}{cfg}{hw}{off}".encode()))
                H, W = hw
                Cm = 2 * Cc if t == "both" else Cc
                steps = torch.tensor([0, 3, 6, 1, 5])
                tab = d.distill_coefficients(steps)
                coef = tab.cuda().contiguous()
                z = torch.randn(B, Cc, H, W, generator=g)
                o1 = torch.randn(B * (2 if cfg else 1), Cm, H, W, generator=g) * 1.5
                o2 = torch.randn(B * (2 if cfg else 1), Cm, H, W, generator=g) * 1.5
                zd, o1d, o2d = _offset(z.cuda(), off), _offset(o1.cuda(), off), _offset(o2.cuda(), off)
                zm, x1 = _offset(torch.zeros(B, Cc, H, W, device="cuda"), off), _offset(torch.zeros(B, Cc, H, W, device="cuda"), off)
                xt, et = _offset(torch.zeros(B, Cc, H, W, device="cuda"), off), _offset(torch.zeros(B, Cc, H, W, device="cuda"), off)
                st = _lib.current_stream_ptr()
                _lib.check(L.vdt_op_distill_step(_lib.ptr(o1d), _lib.ptr(zd), _lib.ptr(zm), _lib.ptr(x1), _lib.ptr(coef), B, Cc, H * W,
                                                 int(cfg), _lib.OUT_TYPES[t], w, st))
                _lib.check(L.vdt_op_distill_target(_lib.ptr(o2d), _lib.ptr(zm), _lib.ptr(x1), _lib.ptr(zd), _lib.ptr(xt), _lib.ptr(et),
                                                   _lib.ptr(coef), B, Cc, H * W, int(cfg), _lib.OUT_TYPES[t], w, st))
                torch.cuda.synchronize()
                c0, c1 = tab[0].double(), tab[1].double()
                col = lambda c, k: c[:, k].reshape(B, 1, 1, 1)          # noqa: E731
                x1w, m1 = _x0_fp64(z, o1, c0, t, w, cfg)
                zmw = col(c0, 6) * z.double() + col(c0, 7) * x1w
                zm_scale = (col(c0, 6) * z.double()).abs() + (col(c0, 7) * x1w).abs() + col(c0, 7).abs() * m1
                # the target kernel from the kernel's own z_t' and x1 (fp32 inputs), so the two kernels are bounded separately
                x2w, m2 = _x0_fp64(zm.cpu(), o2, c1, t, w, cfg)
                x1g = x1.cpu().double()
                xtw = col(c1, 8) * x1g + col(c1, 9) * x2w
                xt_scale = (col(c1, 8) * x1g).abs() + col(c1, 9).abs() * (x2w.abs() + m2)
                etw = z.double() * col(c0, 12) - xtw * col(c0, 13)
                et_scale = (z.double() * col(c0, 12)).abs() + (xt_scale * col(c0, 13)).abs()
                rels = dict(
                    x1=((x1.cpu().double() - x1w).abs() / (m1 + 1e-30)).max().item(),
                    z_mid=((zm.cpu().double() - zmw).abs() / (zm_scale + 1e-30)).max().item(),
                    x_target=((xt.cpu().double() - xtw).abs() / (xt_scale + 1e-30)).max().item(),
                    eps_target=((et.cpu().double() - etw).abs() / (et_scale + 1e-30)).max().item())
                res[f"{t}:cfg{int(cfg)}:{H}x{W}:off{off}"] = max(rels.values())
    return dict(worst=max(res.values()), cases=res)


def closed_form():
    """Gaussian data N(mu, s^2 I), the analytic denoiser as teacher (conditional mean mu_y under CFG), and a student that returns in
    fp64 the exact output of the analytic target x~(z_t): the loss and its gradient vanish at fp32 noise level."""
    mu, s = 0.2, 0.3
    N, B, shape = 4, 8, (8, 3, 8, 8)

    def mean_of(y, rows):
        if y is None:
            return torch.full((rows, 1, 1, 1), mu, dtype=torch.float64)
        return (mu + 0.15 * (y.double().cpu() > 0) * torch.cos(y.double().cpu())).reshape(rows, 1, 1, 1)

    def lam(t):
        return torch.from_numpy(logsnr_schedule(t.double().cpu().numpy(), "cosine", -20., 20.).astype(np.float32)).double()

    def output(out_type, x0, z, l):
        a, sg = torch.sigmoid(l).sqrt(), torch.sigmoid(-l).sqrt()
        eps = (z - a * x0) / sg
        return {"x0": x0, "eps": eps, "v": a * eps - sg * x0, "both": torch.cat([x0, eps], dim=1)}[out_type]

    def teacher_for(out_type):
        def f(z, t, y):
            z = z.double().cpu()
            l = lam(t).reshape(-1, 1, 1, 1)
            a, sg2 = torch.sigmoid(l).sqrt(), torch.sigmoid(-l)
            m = mean_of(y, z.shape[0])
            x0 = m + a * s * s / (a * a * s * s + sg2) * (z - a * m)        # E[x0 | z_t]
            return output(out_type, x0, z, l).float().cuda()
        return f

    res = {}
    g = torch.Generator().manual_seed(3)
    for out_type in ("v", "x0", "eps"):
        for w in (0.0, 1.0):
            d = _diffusion(N, out_type, "snr_trunc")
            x = (mu + s * torch.randn(shape, generator=g))
            noise = torch.randn(shape, generator=g)
            # eps at t = 1 (l = -20) is left out: its x0 = z / alpha - eps e^(-l/2) multiplies the fp32 rounding of the output by
            # e^10, so no fp32 target is exact there
            step = torch.tensor([0, 1, 2, 3, 3, 2, 1, 0]) if out_type != "eps" else torch.tensor([0, 1, 2, 2, 1, 0, 1, 2])
            y = torch.randint(1, 11, (B,), generator=g) if w > 0 else None
            teacher = teacher_for(out_type)

            def student(z, t, yy):
                steps = torch.round(t.double().cpu() * N - 1).long()
                x_t, _, info = ref.distill_targets(lambda a, b, c: teacher(a.cuda(), b, c).cpu(), z.cpu(), steps, None if yy is None else yy.cpu(),
                                                   N=N, model_out_type=out_type, w_guide=w)
                return output(out_type, x_t, z.double().cpu(), info["l"][:, 0].reshape(-1, 1, 1, 1)).float().cuda()
            loss, grad = d.distill_loss(teacher, student, x.cuda(), step, None if y is None else y.cuda(), noise=noise.cuda(),
                                        w_guide=w, return_grad=True)
            torch.cuda.synchronize()
            res[f"{out_type}:w{w}"] = dict(loss_max=loss.abs().max().item(), grad_max=grad.abs().max().item())
    return dict(loss_worst=max(v["loss_max"] for v in res.values()), grad_worst=max(v["grad_max"] for v in res.values()),
                cases=res)


def rel(a, b, floor=0.0):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return ((a - b).norm() / (b.norm() + floor)).item()


def composed(w, steps=3):
    """DistillationStep against the oracle UNet under fp32 autograd on the same draws: loss and every student gradient of one
    step, then three optimizer steps against torch AdamW + clip_grad_norm_ + the reference EMA."""
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    cfg = _cfg(hid=128, mult=(1, 1), nrb=1, attn=(False, True), num_classes=10)
    R, B, N = 16, 4, 4
    sd_t = make_state_dict(cfg, 31)
    teacher, student = _net(cfg, sd_t).eval(), _net(cfg, sd_t).train()
    d = _diffusion(N, "v", "snr_trunc", p_uncond=0.25)
    lr, gn, decay = 2e-4, 1.0, 0.9999
    ds = DistillationStep(student, teacher, d, w_guide=w, lr=lr, grad_norm=gn, use_ema=True, ema_decay=decay)
    ref_p = {k: v.clone().requires_grad_(True) for k, v in sd_t.items()}
    opt = torch.optim.AdamW(list(ref_p.values()), lr=lr, weight_decay=0.0)
    shadow = {k: v.detach().clone() for k, v in ref_p.items()}
    twin = torch.Generator("cuda").manual_seed(8191)                   # replays DistillationStep.draw's stream
    g = torch.Generator().manual_seed(5)
    oracle_teacher = lambda a, b, c: _unet_forward(sd_t, cfg, a.float(), b, c, None)      # noqa: E731
    rec = dict(loss_rel=[], gnorm=[], gnorm_ref=[])
    for it in range(steps):
        x = (torch.rand(B, 3, R, R, generator=g) * 2 - 1)
        y = torch.randint(1, 11, (B,), generator=g)
        step = torch.randint(N, (B,), device="cuda", generator=twin)
        noise = torch.empty(x.shape, device="cuda").normal_(generator=twin)
        keep = torch.rand((B,), device="cuda", generator=twin) >= d.p_uncond
        yk = y * keep.cpu().long() if w == 0 else y
        if it == 0:                                                    # the gradients of this step, from the same draws
            _, first_grads = ds.loss_and_grads(x.cuda(), y.cuda(), step=step, noise=noise, keep=keep)
        loss = ds.step(x.cuda(), y.cuda())                             # draws them again from its own generator (seed 8191)
        rec["gnorm"].append(math.sqrt(float(ds.last_grad_sq)))
        # the reference: fp64 Algorithm 2 over the oracle teacher, then the oracle's train_loss with x0 := x~, noise := eps~
        lt = torch.from_numpy(logsnr_schedule(((step.cpu().double() + 1) / N).numpy(), "cosine", -20., 20.).astype(np.float32))
        lt = lt.reshape(-1, 1, 1, 1)
        z_t = x * torch.sigmoid(lt).sqrt() + noise.cpu() * torch.sigmoid(-lt).sqrt()
        with torch.no_grad():
            x_t, e_t, _ = ref.distill_targets(oracle_teacher, z_t, step.cpu(), yk, N=N, model_out_type="v", w_guide=w)
        t = (step.cpu().double() + 1) / N
        with torch.enable_grad():
            per, _ = oracle_train_loss(lambda a, b, c: _unet_forward(ref_p, cfg, a, b, c, None), x_t.float(), t, yk, e_t.float(),
                                       model_out_type="v", reweight_type="snr_trunc")
            opt.zero_grad(set_to_none=True)
            per.mean().backward()
        rec["loss_rel"].append(abs(float(loss) - float(per.mean())) / abs(float(per.mean())))
        if it == 0:
            errs = {k: rel(first_grads[k], ref_p[k].grad, floor=1e-3 * ref_p[k].grad.norm().item() + 1e-12) for k in sd_t}
            worst = sorted(errs.items(), key=lambda kv: -kv[1])[:5]
        rec["gnorm_ref"].append(float(torch.nn.utils.clip_grad_norm_(list(ref_p.values()), max_norm=gn)))
        opt.step()
        dd = min(decay, (1 + it + 1) / (10 + it + 1))
        with torch.no_grad():
            for k in shadow:
                shadow[k] += (1 - dd) * (ref_p[k] - shadow[k])
    torch.cuda.synchronize()
    upd = torch.cat([(p.detach().cpu() - sd_t[k]).reshape(-1) for k, p in student.named_parameters()]).double()
    upd_ref = torch.cat([(ref_p[k].detach() - sd_t[k]).reshape(-1) for k, _ in student.named_parameters()]).double()
    return dict(grad_rel_worst=worst[0][1], worst=worst, loss_rel_worst=max(rec["loss_rel"]),
                gnorm_rel_worst=max(abs(a - b) / abs(b) for a, b in zip(rec["gnorm"], rec["gnorm_ref"])),
                cosine_of_updates=float((upd @ upd_ref) / (upd.norm() * upd_ref.norm())),
                update_norm_ratio=float(upd.norm() / upd_ref.norm()),
                ema_rel_worst=max(rel(ds.optimizer.shadow[k], shadow[k]) for k in shadow), **rec)


def works(iters=600, teacher_iters=400):
    """A hid-64 unconditional network at 16^2, first trained for a few hundred steps on synthetic data (smooth random colour
    fields) so that it is a denoiser, is distilled from 8 to 4 DDIM steps on the same data: the student's 4-step samples from
    fixed noise against the teacher's 8-step samples, relative to the teacher's own 4-step ones."""
    import time
    from v_diffusion_b200.training import TrainingStep
    cfg = _cfg(hid=64, mult=(1, 2), nrb=1, attn=(False, True), num_classes=0)
    torch.manual_seed(0)
    net = UNet(3, 64, 3, [1, 2], 1, [False, True], num_heads=1).cuda().train()         # the reference's own initialisation
    g = torch.Generator().manual_seed(11)
    base = torch.randn(4096, 3, 4, 4, generator=g)
    data = torch.tanh(torch.nn.functional.interpolate(base, size=(16, 16), mode="bilinear", align_corners=False) * 1.5).cuda()
    d4, d8 = _diffusion(4, "v"), _diffusion(8, "v")
    gi = torch.Generator().manual_seed(12)
    t0 = time.perf_counter()
    ts = TrainingStep(net, _diffusion(1000, "v"), timesteps=0, lr=5e-4, use_ema=False)
    for it in range(teacher_iters):
        ts.step(data[torch.randint(4096, (64,), generator=gi)], None)
    teacher_seconds = time.perf_counter() - t0
    sd = {k: v.detach().cpu().clone() for k, v in net.state_dict().items()}
    teacher, student = _net(cfg, sd).eval(), _net(cfg, sd).train()
    ds = DistillationStep(student, teacher, d4, lr=3e-4, use_ema=False)
    gi = torch.Generator().manual_seed(12)
    losses, t0 = [], time.perf_counter()
    for it in range(iters):
        idx = torch.randint(4096, (32,), generator=gi)
        losses.append(float(ds.step(data[idx], None, lr=3e-4 * (1 - it / iters))))
    seconds = time.perf_counter() - t0
    student.eval()
    noise = torch.randn(64, 3, 16, 16, generator=torch.Generator().manual_seed(13))
    t8 = d8.p_sample(teacher, tuple(noise.shape), noise=noise, device="cuda", use_ddim=True)
    t4 = d4.p_sample(teacher, tuple(noise.shape), noise=noise, device="cuda", use_ddim=True)
    s4 = d4.p_sample(student, tuple(noise.shape), noise=noise, device="cuda", use_ddim=True)
    rms = lambda a, b: (a - b).pow(2).mean().sqrt().item()             # noqa: E731
    k = max(1, iters // 10)
    return dict(student_rms=rms(s4, t8), teacher4_rms=rms(t4, t8), ratio=rms(s4, t8) / rms(t4, t8),
                loss_first=float(np.mean(losses[:k])), loss_last=float(np.mean(losses[-k:])), seconds=seconds, iters=iters,
                teacher_seconds=teacher_seconds, teacher_iters=teacher_iters,
                finite=bool(torch.isfinite(s4).all()))


def driver():
    """python -m v_diffusion_b200.distill for 2 stages x 3 iterations on a 64-image synthetic .npy: stage 2's teacher equals
    stage 1's EMA shadow bit for bit, and student_N.pt loads through generate.load_reference_checkpoint and samples at T = N."""
    import v_diffusion_b200.training as training
    from v_diffusion_b200 import distill, build_from_config
    from v_diffusion_b200.generate import load_reference_checkpoint
    seen = []

    class Recording(training.DistillationStep):
        def __init__(self, student, teacher, *a, **kw):
            seen.append({k: p.detach().cpu().clone() for k, p in teacher.named_parameters()})
            super().__init__(student, teacher, *a, **kw)
    config = {"data": {"name": "cifar10"}, "conditional": {"p_uncond": 0.1, "use_cfg": True, "w_guide": 0.0},
              "diffusion": {"allow_rescale": False, "intp_frac": 0.0, "logsnr_max": 20.0, "logsnr_min": -20.0,
                            "logsnr_schedule": "cosine", "loss_type": "mse", "model_out_type": "v", "model_var_type": "fixed_large",
                            "reweight_type": "snr_trunc", "sample_timesteps": 8, "train_timesteps": 0, "x0eps_coef": False},
              "model": {"apply_attn": [False, True], "ch_multipliers": [1, 2], "drop_rate": 0.0, "embedding_dim": 256,
                        "hid_channels": 64, "in_channels": 3, "num_heads": 1, "num_res_blocks": 1}}
    cfg = _cfg(hid=64, mult=(1, 2), nrb=1, attn=(False, True), num_classes=10)
    res = {}
    with tempfile.TemporaryDirectory() as tmp:
        g = np.random.default_rng(0)
        np.save(os.path.join(tmp, "x.npy"), g.integers(0, 256, (64, 32, 32, 3), dtype=np.uint8))
        np.save(os.path.join(tmp, "y.npy"), g.integers(1, 11, (64,)).astype(np.int64))
        with open(os.path.join(tmp, "c.json"), "w") as f:
            json.dump(config, f)
        torch.save({"model": make_state_dict(cfg, 41)}, os.path.join(tmp, "t.pt"))
        out = os.path.join(tmp, "out")
        saved, training.DistillationStep = training.DistillationStep, Recording
        try:
            distill.main(["--config-path", os.path.join(tmp, "c.json"), "--ckpt-path", os.path.join(tmp, "t.pt"),
                          "--images", os.path.join(tmp, "x.npy"), "--labels", os.path.join(tmp, "y.npy"), "--teacher-steps", "8",
                          "--stages", "2", "--iters", "3", "--batch-size", "8", "--lr", "1e-4", "--out-dir", out])
        finally:
            training.DistillationStep = saved
        c4 = torch.load(os.path.join(out, "student_4.pt"), map_location="cpu")
        sd4, use_cfg = load_reference_checkpoint(os.path.join(out, "student_4.pt"), use_ema=True)
        res["stages_seen"] = len(seen)
        res["stage2_teacher_is_stage1_ema"] = len(seen) == 2 and all(torch.equal(seen[1][k], sd4[k]) for k in seen[1])
        res["stage1_teacher_is_ckpt"] = all(torch.equal(seen[0][k], make_state_dict(cfg, 41)[k]) for k in seen[0])
        res["ema_differs_from_teacher"] = any(not torch.equal(seen[1][k], seen[0][k]) for k in seen[0])
        res["keys"] = dict(sample_timesteps=c4.get("sample_timesteps"), distill_w_guide=c4.get("distill_w_guide"),
                           has_optimizer="optimizer" in c4, has_ema="ema" in c4)
        res["student_2_exists"] = os.path.exists(os.path.join(out, "student_2.pt"))
        diffusion, model, chw = build_from_config(config, use_cfg, 0.0, 4)
        model.load_state_dict(sd4)
        model = model.cuda().eval()
        x = diffusion.p_sample(model, (4,) + chw, label=torch.tensor([1, 2, 3, 0]), device="cuda", seed=1, use_ddim=True)
        res["sample_finite"] = bool(torch.isfinite(x).all())
        res["sample_shape"] = list(x.shape)
    return res


def main():
    torch.cuda.set_device(0)
    mode = sys.argv[1]
    if mode == "kernels":
        out = kernels()
    elif mode == "closed_form":
        out = closed_form()
    elif mode == "composed":
        out = composed(float(sys.argv[2]))
    elif mode == "works":
        out = works()
    elif mode == "driver":
        out = driver()
    else:
        raise SystemExit(f"unknown mode {mode}")
    print("RESULT " + json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
