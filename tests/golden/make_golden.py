"""Generate the golden fixtures in this directory FROM THE UNMODIFIED REFERENCE.

Run in the build container only (needs /root/reference):

    python tests/golden/make_golden.py

It imports tqch/v-diffusion-torch from /root/reference (matplotlib stubbed, SURVEY §10.3),
loads the oracle's deterministic synthetic state_dict into the reference's own ``UNet`` (strict
load: proves the key/shape layout), runs ``UNet.forward`` and ``GaussianDiffusion.p_sample`` on
seeded inputs and stores inputs + outputs as .npz.  The fixtures pin ``oracle/`` (CPU tests) and
the CUDA path (gpu tests); the GPU box never sees /root/reference.
"""
import json
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF = "/root/reference"

_m = types.ModuleType("matplotlib"); _m.rcParams = {}
sys.modules.setdefault("matplotlib", _m)
sys.modules.setdefault("matplotlib.pyplot", types.ModuleType("matplotlib.pyplot"))
sys.path.insert(0, REF)
from v_diffusion import UNet, GaussianDiffusion, get_logsnr_schedule, fill_with_defaults  # noqa: E402
from v_diffusion.diffusion import logsnr_to_posterior, logsnr_to_posterior_ddim  # noqa: E402
from v_diffusion.functions import get_timestep_embedding  # noqa: E402

from oracle.unet_ref import make_state_dict, state_dict_shapes  # noqa: E402
from tests.cases import (UNET_CASES, SAMPLE_CASES, FULL_CASES, TRAIN_CASES, build_inputs, build_sample_inputs,  # noqa: E402
                         build_full_inputs, full_state_dict, build_train_inputs, golden_sample_index)

torch.set_num_threads(os.cpu_count())


def ref_unet(cfg, seed):
    net = UNet(cfg["in_channels"], cfg["hid_channels"], cfg["out_channels"], cfg["ch_multipliers"],
               cfg["num_res_blocks"], cfg["apply_attn"], embedding_dim=cfg["embedding_dim"],
               head_dim=cfg["head_dim"], num_heads=cfg["num_heads"], num_classes=cfg["num_classes"],
               multitags=cfg["multitags"])
    ref_shapes = {k: tuple(v.shape) for k, v in net.state_dict().items()}
    assert ref_shapes == state_dict_shapes(cfg), "state_dict layout mismatch vs reference"
    net.load_state_dict(make_state_dict(cfg, seed), strict=True)
    return net.eval()


def main():
    # ---- UNet forward goldens
    for name, case in UNET_CASES.items():
        cfg = case["cfg"]
        net = ref_unet(cfg, case["seed"])
        x, t, y = build_inputs(case)
        feats = {}
        hooks = []
        for mod_name in case.get("trace", []):
            mod = net.get_submodule(mod_name)
            hooks.append(mod.register_forward_hook(
                lambda m, i, o, n=mod_name: feats.__setitem__(n, o.detach().clone())))
        with torch.no_grad():
            out = net(x, t, y)
        for h in hooks:
            h.remove()
        arrs = {"out": out.numpy()}
        for k, v in feats.items():
            v = v.numpy()
            if case.get("trace_keep"):                  # a seeded sample of the feature map keeps the fixture small
                idx = golden_sample_index(v.size, case["trace_keep"], "trace:" + k)
                arrs["trace_index:" + k], v = idx, v.reshape(-1)[idx]
            arrs["trace:" + k] = v
        np.savez_compressed(os.path.join(HERE, f"unet_{name}.npz"), **arrs)
        print(name, tuple(out.shape), float(out.abs().mean()), float(out.abs().max()))

    # ---- sampler goldens
    for name, case in SAMPLE_CASES.items():
        cfg = UNET_CASES[case["unet"]]["cfg"]
        net = ref_unet(cfg, UNET_CASES[case["unet"]]["seed"])
        noise, label, step_noise = build_sample_inputs(case, cfg)
        logsnr_fn = get_logsnr_schedule("cosine", -20., 20., rescale=False)
        diff = GaussianDiffusion(
            logsnr_fn=logsnr_fn, sample_timesteps=case["T"], model_out_type=case["model_out_type"],
            model_var_type=case["var_type"], reweight_type="snr_trunc", loss_type="mse",
            intp_frac=case.get("intp_frac"), w_guide=case["w_guide"], x0eps_coef=case.get("x0eps_coef", False))
        outs = []

        def rec(x, t, y):
            o = net(x, t, y)
            outs.append(o.clone())
            return o
        # the reference draws one normal_ per step from Generator(seed) (diffusion.py:389);
        # build_sample_inputs replays exactly that sequence into step_noise.
        x = diff.p_sample(rec, shape=tuple(noise.shape), noise=noise, label=label, device="cpu",
                          seed=case["seed"], use_ddim=case["use_ddim"])
        np.savez_compressed(os.path.join(HERE, f"sample_{name}.npz"), out=x.numpy(),
                            model_out=torch.stack(outs).numpy())
        print(name, tuple(x.shape), float(x.abs().mean()), float(x.abs().max()))

    # ---- p_sample_progressive (diffusion.py:416-441): fp32 step tensor (:421), x0 previews every pred_freq steps
    for name, pred_freq in (("ddim_cfg_v", 3), ("ancestral_cfg_v", 16)):
        case = SAMPLE_CASES[name]
        cfg = UNET_CASES[case["unet"]]["cfg"]
        net = ref_unet(cfg, UNET_CASES[case["unet"]]["seed"])
        noise, label, step_noise = build_sample_inputs(case, cfg)
        diff = GaussianDiffusion(
            logsnr_fn=get_logsnr_schedule("cosine", -20., 20., rescale=False), sample_timesteps=case["T"],
            model_out_type=case["model_out_type"], model_var_type=case["var_type"], reweight_type="snr_trunc",
            loss_type="mse", intp_frac=case.get("intp_frac"), w_guide=case["w_guide"])
        x, preds = diff.p_sample_progressive(net, shape=tuple(noise.shape), noise=noise, label=label, device="cpu",
                                             seed=case["seed"], use_ddim=case["use_ddim"], pred_freq=pred_freq)
        np.savez_compressed(os.path.join(HERE, f"progressive_{name}.npz"), out=x.numpy(), preds=preds.numpy(),
                            pred_freq=np.int64(pred_freq))
        print("progressive", name, tuple(x.shape), tuple(preds.shape), float(x.abs().max()))

    # ---- full-length trajectories of the real CIFAR-10 networks (BASELINE configs[0], configs[1] at B=8)
    from v_diffusion_b200.unet import UNet as OurUNet
    for name, case in FULL_CASES.items():
        cfg = case["cfg"]
        sd, net = full_state_dict(case, UNet)
        sd_ours, _ = full_state_dict(case, OurUNet)
        assert list(sd) == list(sd_ours) and all(torch.equal(sd[k], sd_ours[k]) for k in sd), \
            "this package's UNet constructor no longer reproduces the reference's initialisation"
        net.load_state_dict(sd, strict=True)
        net.eval()
        noise, label = build_full_inputs(case)
        diff = GaussianDiffusion(
            logsnr_fn=get_logsnr_schedule("cosine", -20., 20., rescale=False), sample_timesteps=case["T"],
            model_out_type=case["model_out_type"], model_var_type=case["var_type"], reweight_type="snr_trunc",
            loss_type="mse", intp_frac=case["intp_frac"], w_guide=case["w_guide"])
        outs = []
        keep = case["keep_rows"]

        def rec(x, t, y):
            o = net(x, t, y)
            outs.append(o[:keep].clone())
            return o
        import time
        t0 = time.time()
        x = diff.p_sample(rec, shape=tuple(noise.shape), noise=noise, label=label, device="cpu",
                          seed=case["noise_seed"], use_ddim=case["use_ddim"])
        mo = torch.stack(outs)
        idx = golden_sample_index(mo[0].numel(), case["keep_entries"], f"full_{name}")
        np.savez_compressed(os.path.join(HERE, f"full_{name}.npz"), out=x.numpy(), model_out=mo.reshape(len(mo), -1)[:, torch.from_numpy(idx).long()].numpy(),
                            model_out_index=idx)
        print("full", name, tuple(x.shape), tuple(mo.shape), float(x.abs().mean()), float(x.abs().max()),
              f"{time.time() - t0:.1f}s")

    # ---- train_loss (diffusion.py:492-545): x_t, per-sample loss, d loss.mean() / d model_out by the reference's autograd
    for name, case in TRAIN_CASES.items():
        cfg = UNET_CASES[case["unet"]]["cfg"]
        net = ref_unet(cfg, UNET_CASES[case["unet"]]["seed"])
        x0, t, noise, y = build_train_inputs(case, cfg)
        diff = GaussianDiffusion(
            logsnr_fn=get_logsnr_schedule("cosine", -20., 20., rescale=False), sample_timesteps=1000,
            model_out_type=case["model_out_type"], model_var_type="fixed_large", reweight_type=case["reweight_type"],
            loss_type="mse", p_uncond=0.1)
        seen = {}

        def fn(x_t, tt, yy):
            with torch.no_grad():
                o = net(x_t, tt, None if yy is None else yy.clone())
            o = o.detach().requires_grad_(True)
            seen["x_t"], seen["out"] = x_t.detach().clone(), o
            return o
        torch.manual_seed(case["seed"])                 # the p_uncond mask is drawn from the global CPU generator (:527-529)
        yy = None if y is None else y.clone()
        loss = diff.train_loss(fn, x_0=x0, t=t, y=yy, noise=noise)
        loss.mean().backward()
        np.savez_compressed(os.path.join(HERE, f"train_{name}.npz"), x_t=seen["x_t"].numpy(), model_out=seen["out"].detach().numpy(),
                            loss=loss.detach().numpy(), grad_out=seen["out"].grad.numpy(),
                            y_after=(yy.numpy() if yy is not None else np.zeros(0)))
        print("train", name, loss.detach().numpy())

    # ---- coefficient known answers (T = 100, cosine +-20) straight from the reference functions
    T = 100
    logsnr_fn = get_logsnr_schedule("cosine", -20., 20., rescale=False)
    step = torch.arange(T, dtype=torch.float64)
    ls = logsnr_fn(step / T).to(torch.float32).reshape(-1, 1, 1, 1)
    lt = logsnr_fn((step + 1) / T).to(torch.float32).reshape(-1, 1, 1, 1)
    co = {"logsnr_s": ls.flatten().numpy(), "logsnr_t": lt.flatten().numpy()}
    c1, c2, _ = logsnr_to_posterior_ddim(ls, lt, eta=0.)
    co["ddim_c1"], co["ddim_c2"] = c1.flatten().numpy(), c2.flatten().numpy()
    for vt in ("fixed_small", "fixed_large", "fixed_medium"):
        c1, c2, lv = logsnr_to_posterior(ls, lt, vt, intp_frac=0.3)
        co[f"{vt}_c1"], co[f"{vt}_c2"], co[f"{vt}_logvar"] = (
            c1.flatten().numpy(), c2.flatten().numpy(), lv.flatten().numpy())
    # x0eps_coef=True variants (diffusion.py:137-140, 180-182; the DDIM pair comes back un-exponentiated)
    c1, c2, _ = logsnr_to_posterior_ddim(ls, lt, eta=0., x0eps_coef=True)
    co["x0eps_ddim_c1"], co["x0eps_ddim_c2"] = c1.flatten().numpy(), c2.flatten().numpy()
    c1, c2, lv = logsnr_to_posterior(ls, lt, "fixed_small", x0eps_coef=True)
    co["x0eps_small_c1"], co["x0eps_small_c2"], co["x0eps_small_logvar"] = (
        c1.flatten().numpy(), c2.flatten().numpy(), lv.flatten().numpy())
    co["alpha_t"] = torch.sigmoid(lt).sqrt().flatten().numpy()
    co["sigma_t"] = torch.sigmoid(-lt).sqrt().flatten().numpy()
    tt = torch.tensor([0.37, 0.01, 1.0, 0.5], dtype=torch.float64)
    co["temb_t"] = tt.numpy()
    co["temb_256"] = get_timestep_embedding(tt, 256).numpy()
    co["temb_64"] = get_timestep_embedding(tt, 64).numpy()
    # every schedule get_logsnr_schedule knows (diffusion.py:52-96), T = 50, default +-20 range
    for sched in ("cosine", "linear", "sigmoid", "legacy"):
        fn = get_logsnr_schedule(sched, -20., 20., rescale=False)
        st = torch.arange(50, dtype=torch.float64)
        ls_, lt_ = fn(st / 50).to(torch.float32), fn((st + 1) / 50).to(torch.float32)
        co[f"{sched}_logsnr_s"], co[f"{sched}_logsnr_t"] = ls_.numpy(), lt_.numpy()
        c1_, c2_, lv_ = logsnr_to_posterior(ls_, lt_, "fixed_large")
        co[f"{sched}_c1"], co[f"{sched}_c2"], co[f"{sched}_logvar"] = c1_.numpy(), c2_.numpy(), lv_.numpy()
    np.savez_compressed(os.path.join(HERE, "coefs_T100.npz"), **co)

    # ---- config merge known answer (utils.py:193-201 on the shipped JSONs)
    merged = {}
    for n in ("cifar10_cond", "cifar10_uncond", "celeba"):
        with open(f"{REF}/configs/{n}.json") as f:
            c = json.load(f)
        with open(f"{REF}/configs/defaults.json") as f:
            d = json.load(f)
        fill_with_defaults(c, d)
        merged[n] = {"model": c["model"], "diffusion": c["diffusion"], "conditional": c["conditional"]}
    with open(os.path.join(HERE, "merged_configs.json"), "w") as f:
        json.dump(merged, f, indent=1, sort_keys=True)
    print("done")


if __name__ == "__main__":
    main()
