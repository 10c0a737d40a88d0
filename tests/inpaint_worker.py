"""Child process of tests/test_inpaint_gpu.py: one whole-network inpainting case on cuda:0.  Prints one JSON line.

    python -m tests.inpaint_worker parity ddim_cfg_v 12 fp16 dpmpp_2m
    python -m tests.inpaint_worker progressive ddim_cfg_v 20 fp16x3
    python -m tests.inpaint_worker exactness
"""
import ctypes as C
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import unet_forward, make_state_dict                                       # noqa: E402
from tests.cases import UNET_CASES, SAMPLE_CASES, build_sample_inputs                  # noqa: E402
from tests.dpm_solver_worker import _model                                             # noqa: E402
from tests.inpaint_ref import p_sample as ref_p_sample                                 # noqa: E402
from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule, _lib              # noqa: E402

CASES = {
    "ddim_cfg_v": SAMPLE_CASES["ddim_cfg_v"],                  # small_cond, v-prediction, CFG w = 1
    "ddim_cfg_multitag": SAMPLE_CASES["ddim_cfg_multitag"],    # small_multitag, CFG w = 1 on multi-hot labels
    # small_hd64_x0 (unconditional, x0-prediction) under ancestral sampling with injected step noise
    "ancestral_x0": dict(SAMPLE_CASES["ddim_x0_uncond"], use_ddim=False, var_type="fixed_large", seed=28),
}


def _diffusion(case, T):
    return GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), T, case["model_out_type"], case["var_type"],
                             "snr_trunc", "mse", intp_frac=case.get("intp_frac"), w_guide=case["w_guide"])


def inpaint_inputs(shape, T, seed):
    """known in [-1, 1]; a mask whose left half is 1 and whose right half is a random soft mask with exact zeros; z'."""
    g = torch.Generator().manual_seed(seed)
    known = torch.rand(shape, generator=g) * 2 - 1
    soft = torch.rand(shape, generator=g)
    soft = torch.where(soft < 0.3, torch.zeros_like(soft), soft)
    mask = soft.clone()
    mask[..., : shape[3] // 2] = 1.0
    known_noise = torch.randn((T,) + tuple(shape), generator=g)
    return known, mask, known_noise


def _setup(name, T, operand):
    case = dict(CASES[name], T=T)
    ucase = UNET_CASES[case["unet"]]
    cfg = ucase["cfg"]
    noise, label, step_noise = build_sample_inputs(case, cfg)
    sd = make_state_dict(cfg, ucase["seed"])
    oracle_net = lambda x, t, y: unet_forward(sd, cfg, x, t, y)                         # noqa: E731
    known, mask, known_noise = inpaint_inputs(tuple(noise.shape), T, case["seed"] + 3000)
    return (case, cfg, noise, label, step_noise if not case["use_ddim"] else None, oracle_net, _model(cfg, ucase["seed"], operand),
            _diffusion(case, T), known, mask, known_noise)


def parity(name, T, operand, solver):
    """Fused and generic-callable inpainting against the reference loop over the oracle UNet (injected z')."""
    solver = None if solver == "none" else solver
    case, cfg, noise, label, step_noise, oracle_net, net, diff, known, mask, known_noise = _setup(name, T, operand)
    shape = tuple(noise.shape)
    kw = dict(use_ddim=case["use_ddim"], step_noise=step_noise, solver=solver)
    rec_ref = []
    ref = ref_p_sample(oracle_net, shape, noise, label, T=T, model_out_type=case["model_out_type"], w_guide=case["w_guide"],
                       var_type=case["var_type"], intp_frac=case.get("intp_frac"), record=rec_ref, known=known, mask=mask,
                       known_noise=known_noise, **kw)
    fused = diff.p_sample(net, shape, noise=noise, label=label, device="cuda", known=known, mask=mask, known_noise=known_noise, **kw)
    plain = diff.p_sample(net, shape, noise=noise, label=label, device="cuda", **kw)
    rec = []

    def wrapped(x, t, y):
        o = net(x, t, y)
        rec.append(o.cpu())
        return o
    generic = diff.p_sample(wrapped, shape, noise=noise, label=label, device="cuda", known=known, mask=mask,
                            known_noise=known_noise, **kw)
    step_rel = [((o - r).norm() / r.norm()).item() for o, (_, r) in zip(rec, rec_ref)]
    # z' from the library's stream (no known_noise): the fused and generic paths draw the same z' for the same seed
    fused_s = diff.p_sample(net, shape, noise=noise, label=label, device="cuda", seed=11, known=known, mask=mask, **kw)
    generic_s = diff.p_sample(lambda x, t, y: net(x, t, y), shape, noise=noise, label=label, device="cuda", seed=11, known=known,
                              mask=mask, **kw)
    ones = mask == 1
    return dict(fused_max_abs=(fused - ref).abs().max().item(), generic_max_abs=(generic - ref).abs().max().item(),
                fused_vs_generic=(fused - generic).abs().max().item(), steps=len(rec), worst_step_rel=max(step_rel),
                seeded_fused_vs_generic=(fused_s - generic_s).abs().max().item(),
                ones_equal=torch.equal(fused[ones], known[ones]) and torch.equal(generic[ones], known[ones]),
                differs_from_plain=(fused - plain).abs().max().item(),
                finite=bool(torch.isfinite(fused).all() and torch.isfinite(fused_s).all()))


def progressive(name, T, operand):
    """p_sample_progressive with inpainting (several range calls) against the reference's progressive loop."""
    case, cfg, noise, label, step_noise, oracle_net, net, diff, known, mask, known_noise = _setup(name, T, operand)
    shape = tuple(noise.shape)
    pred_freq = 3
    res = dict(w_guide=case["w_guide"])
    for solver in (None, "dpmpp_2m"):
        preds_ref = []
        ref = ref_p_sample(oracle_net, shape, noise, label, T=T, model_out_type=case["model_out_type"], w_guide=case["w_guide"],
                           use_ddim=True, pred_record=preds_ref, t_fp32=True, solver=solver, known=known, mask=mask,
                           known_noise=known_noise)
        x, preds = diff.p_sample_progressive(net, shape, noise=noise, label=label, device="cuda", use_ddim=True,
                                             pred_freq=pred_freq, solver=solver, known=known, mask=mask, known_noise=known_noise)
        want = torch.stack([p for ti, p in preds_ref if (ti + 1) % pred_freq == 0][::-1][:T // pred_freq])
        tag = solver or "ddim"
        res[f"{tag}_final_max_abs"] = (x - ref).abs().max().item()
        res[f"{tag}_previews_max_abs"] = (preds - want).abs().max().item()
        res[f"{tag}_previews"] = int(preds.shape[0])
    return res


def _range(net, sc, x, label, first, num, pred, inpaint):
    plan = net.plan_for(x.shape[2], torch.device("cuda", 0))
    _lib.check(_lib.lib().vdt_p_sample_range_inpaint(plan, C.byref(sc), C.byref(inpaint), _lib.ptr(x), _lib.ptr(label), None,
                                                     x.shape[0], first, num, _lib.ptr(pred), _lib.current_stream_ptr()))
    torch.cuda.synchronize()


def exactness():
    """Bit-identical properties of fused inpainting on small_cond with CFG (w = 1, v-prediction)."""
    case = SAMPLE_CASES["ddim_cfg_v"]
    ucase = UNET_CASES[case["unet"]]
    cfg = ucase["cfg"]
    T = 12
    diff = _diffusion(case, T)
    g = torch.Generator().manual_seed(41)
    B = 7
    shape = (B, 3, 16, 16)
    noise = torch.randn(shape, generator=g)
    label = torch.randint(0, 11, (B,), generator=g)
    known, mask, known_noise = inpaint_inputs(shape, T, 42)
    known2, mask2, _ = inpaint_inputs(shape, T, 43)
    net = _model(cfg, ucase["seed"])
    res = {}

    def run(model, solver, use_ddim=True, seed=5, **kw):
        return diff.p_sample(model, shape, noise=noise, label=label, device="cuda", use_ddim=use_ddim, seed=seed, solver=solver, **kw)
    # (1) m = 0 equals the call without inpainting (DDIM, 2M and ancestral; z' from the stream and injected)
    res["mask0_equal"] = all(torch.equal(run(net, s, u, known=known, mask=torch.zeros(shape), **kw), run(net, s, u))
                             for s, u in ((None, True), ("dpmpp_2m", True), (None, False))
                             for kw in ({}, {"known_noise": known_noise}))
    # (2) pixels with m = 1 come out equal to known; the stream is a function of the seed
    full = run(net, "dpmpp_2m", known=known, mask=mask)
    ones = mask == 1
    res["ones_equal"] = torch.equal(full[ones], known[ones])
    res["same_seed_equal"] = torch.equal(full, run(net, "dpmpp_2m", known=known, mask=mask))
    res["other_seed_differs"] = (full - run(net, "dpmpp_2m", seed=6, known=known, mask=mask)).abs().max().item()
    # (3) several chunks over two lanes and a ragged last chunk (7 images, 2 per chunk under CFG) vs one chunk
    chunked = _model(cfg, ucase["seed"], max_rows=4)
    res["chunked_max_abs"] = (run(chunked, "dpmpp_2m", known=known, mask=mask) - full).abs().max().item()
    res["chunked_equal"] = res["chunked_max_abs"] == 0.0
    res["ddim_chunked_equal"] = torch.equal(run(chunked, None), run(net, None))          # the existing sampler's property
    # (4) split range calls carrying pred_x0 under 2M equal one call; a plain first step on the same exec in between
    sc = diff.sampler_config(True, seed=5, solver="dpmpp_2m")
    kd, md = known.cuda(), mask.cuda()
    ip = _lib.Inpaint(_lib.ptr(kd), _lib.ptr(md), None)
    none = _lib.Inpaint(None, None, None)
    labc = label.cuda()
    x, pred = noise.cuda().clone(), torch.empty(shape, device="cuda")
    first = T - 1
    for n in (1, 4, 2, 3, 2):
        _range(net, sc, x, labc, first, n, pred, ip)
        _range(net, sc, torch.full_like(x, float("nan")), labc, T - 1, 1, None, none)
        first -= n
    assert first == -1
    res["split_equal"] = torch.equal(x.cpu(), full)
    # (5) a cached exec called with another known / mask, then without inpainting, returns what a fresh plan returns
    other = run(net, "dpmpp_2m", known=known2, mask=mask2)
    plain = run(net, "dpmpp_2m")
    fresh_other = run(_model(cfg, ucase["seed"]), "dpmpp_2m", known=known2, mask=mask2)
    fresh_plain = run(_model(cfg, ucase["seed"]), "dpmpp_2m")
    res["repeat_fresh_equal"] = torch.equal(other, fresh_other) and torch.equal(plain, fresh_plain)
    res["finite"] = bool(torch.isfinite(full).all() and torch.isfinite(other).all())
    return res


def main():
    torch.cuda.set_device(0)
    mode = sys.argv[1]
    if mode == "parity":
        out = parity(sys.argv[2], int(sys.argv[3]), sys.argv[4], sys.argv[5])
    elif mode == "progressive":
        out = progressive(sys.argv[2], int(sys.argv[3]), sys.argv[4])
    elif mode == "exactness":
        out = exactness()
    else:
        raise SystemExit(f"unknown mode {mode}")
    print("RESULT " + json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
