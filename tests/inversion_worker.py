"""Child process of tests/test_inversion_gpu.py: one whole-network DDIM-inversion case on cuda:0.  Prints one JSON line.

    python -m tests.inversion_worker parity ddim_cfg_v 10 fp16
    python -m tests.inversion_worker exactness
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
from tests.dpm_solver_worker import _diffusion, _model                                 # noqa: E402
from tests.inversion_ref import ddim_invert as ref_invert, p_sample_from as ref_sample_from   # noqa: E402
from v_diffusion_b200 import _lib                                                      # noqa: E402


def _rel(a, b):
    return ((a - b).norm() / b.norm()).item()


def parity(name, T, operand):
    """Fused and generic-callable inversion against the reference inversion over the oracle UNet, then sampling from a
    halfway latent (p_sample(start_step=T//2)) against the reference start-k loop.  Images come from the case's noise
    squashed into [-1, 1]."""
    case = SAMPLE_CASES[name]
    ucase = UNET_CASES[case["unet"]]
    cfg = ucase["cfg"]
    noise, label, _ = build_sample_inputs(case, cfg)
    x0 = torch.tanh(noise)
    sd = make_state_dict(cfg, ucase["seed"])
    oracle_net = lambda x, t, y: unet_forward(sd, cfg, x, t, y)                         # noqa: E731
    net = _model(cfg, ucase["seed"], operand)
    diff = _diffusion(case, T)
    w, out_type = case["w_guide"], case["model_out_type"]
    rec_ref = []
    ref = ref_invert(oracle_net, x0, label, T=T, model_out_type=out_type, w_guide=w, record=rec_ref)
    fused = diff.ddim_invert(net, x0, label=label)
    rec = []

    def wrapped(x, t, y):
        o = net(x, t, y)
        rec.append(o.cpu())
        return o
    generic = diff.ddim_invert(wrapped, x0, label=label)
    step_rel = [_rel(o, r) for o, (_, r) in zip(rec, rec_ref)]
    # sampling from the middle of the trajectory: both sides start from the fused halfway latent
    k = T // 2
    x_k = diff.ddim_invert(net, x0, label=label, num_steps=k)
    srec_ref = []
    sref = ref_sample_from(oracle_net, x_k, label, T=T, start_step=k, model_out_type=out_type, w_guide=w, record=srec_ref)
    sfused = diff.p_sample(net, tuple(x_k.shape), noise=x_k, label=label, device="cuda", use_ddim=True, start_step=k)
    srec = []

    def swrapped(x, t, y):
        o = net(x, t, y)
        srec.append(o.cpu())
        return o
    sgeneric = diff.p_sample(swrapped, tuple(x_k.shape), noise=x_k, label=label, device="cuda", use_ddim=True, start_step=k)
    sstep_rel = [_rel(o, r) for o, (_, r) in zip(srec, srec_ref)]
    scale = ref.abs().max().item()
    return dict(steps=len(rec), latent_max=scale, fused_max_abs=(fused - ref).abs().max().item(),
                generic_max_abs=(generic - ref).abs().max().item(), fused_rel=(fused - ref).abs().max().item() / scale,
                generic_rel=(generic - ref).abs().max().item() / scale, fused_vs_generic=(fused - generic).abs().max().item() / scale,
                worst_step_rel=max(step_rel), finite=bool(torch.isfinite(fused).all() and torch.isfinite(generic).all()),
                sample_steps=len(srec), sample_fused_max_abs=(sfused - sref).abs().max().item(),
                sample_generic_max_abs=(sgeneric - sref).abs().max().item(),
                sample_fused_vs_generic=(sfused - sgeneric).abs().max().item(), sample_worst_step_rel=max(sstep_rel))


def _invert_range(net, sc, x, label, first, num):
    plan = net.plan_for(x.shape[2], torch.device("cuda", 0))
    _lib.check(_lib.lib().vdt_ddim_invert_range(plan, C.byref(sc), _lib.ptr(x), _lib.ptr(label), x.shape[0], first, num,
                                                _lib.current_stream_ptr()))
    torch.cuda.synchronize()


def _sample_range(net, sc, x, label, step_noise, first, num, pred=None):
    plan = net.plan_for(x.shape[2], torch.device("cuda", 0))
    _lib.check(_lib.lib().vdt_p_sample_range(plan, C.byref(sc), _lib.ptr(x), _lib.ptr(label), _lib.ptr(step_noise), x.shape[0],
                                             first, num, _lib.ptr(pred), _lib.current_stream_ptr()))
    torch.cuda.synchronize()


def exactness():
    """Bit-identical properties of the fused inversion and of sampling from step k, on small_cond with CFG (w = 1, v)."""
    case = SAMPLE_CASES["ddim_cfg_v"]
    ucase = UNET_CASES[case["unet"]]
    cfg = ucase["cfg"]
    T, k = 12, 5
    diff = _diffusion(case, T)
    g = torch.Generator().manual_seed(41)
    B = 7
    shape = (B, 3, 16, 16)
    x0 = torch.rand(shape, generator=g) * 2 - 1
    x0b = torch.rand(shape, generator=g) * 2 - 1
    label = torch.randint(0, 11, (B,), generator=g)
    sn = torch.randn((T,) + shape, generator=g)
    res = {}
    net = _model(cfg, ucase["seed"])
    labc = label.cuda()
    sc = diff.sampler_config(True)
    # (1) inversion [0, k) then [k, T) == [0, T) in one call (and == ddim_invert)
    full = diff.ddim_invert(net, x0, label=label)
    x = x0.cuda().clone()
    _invert_range(net, sc, x, labc, 0, k)
    _invert_range(net, sc, x, labc, k, T - k)
    res["split_equal"] = torch.equal(x.cpu(), full)
    # (2) a cached inversion exec reused after sampling on the same plan == a fresh plan
    diff.p_sample(net, shape, noise=full, label=label, device="cuda", use_ddim=True)
    other = diff.ddim_invert(net, x0b, label=label)
    fresh = diff.ddim_invert(_model(cfg, ucase["seed"]), x0b, label=label)
    again = diff.ddim_invert(net, x0, label=label)
    res["repeat_fresh_equal"] = torch.equal(other, fresh) and torch.equal(again, full)
    # (3) start_step = T is p_sample, for DDIM, ancestral sampling (injected noise and seeded), 2M and inpainting
    mask = (torch.rand((B, 1, 16, 16), generator=g) > 0.5).float()
    eq = []
    for kw in (dict(use_ddim=True), dict(use_ddim=False, step_noise=sn), dict(use_ddim=False, seed=9),
               dict(use_ddim=True, solver="dpmpp_2m"), dict(use_ddim=True, known=x0, mask=mask, seed=3)):
        a = diff.p_sample(net, shape, noise=full, label=label, device="cuda", **kw)
        b = diff.p_sample(net, shape, noise=full, label=label, device="cuda", start_step=T, **kw)
        eq.append(torch.equal(a, b))
    res["start_T_equal"] = eq
    # (4) start_step = k under DDIM and ancestral sampling == vdt_p_sample_range(first_step = k-1, num_steps = k)
    x_k = diff.ddim_invert(net, x0, label=label, num_steps=k)
    eq = []
    for use_ddim, noise_kw in ((True, {}), (False, dict(step_noise=sn)), (False, dict(seed=77))):
        got = diff.p_sample(net, shape, noise=x_k, label=label, device="cuda", use_ddim=use_ddim, start_step=k, **noise_kw)
        scr = diff.sampler_config(use_ddim, seed=noise_kw.get("seed"))
        x = x_k.cuda().clone()
        stn = noise_kw["step_noise"].cuda() if "step_noise" in noise_kw else None
        _sample_range(net, scr, x, labc, stn, k - 1, k)
        eq.append(torch.equal(got, x.cpu()))
    res["start_k_equal_range"] = eq
    # (5) under 2M the first step from k is a DDIM step: one DDIM step from k-1 (its guided x0 into pred), then 2M ranges
    #     carrying pred, equal p_sample(start_step=k, solver="dpmpp_2m")
    got = diff.p_sample(net, shape, noise=x_k, label=label, device="cuda", use_ddim=True, solver="dpmpp_2m", start_step=k)
    x, pred = x_k.cuda().clone(), torch.empty(shape, device="cuda")
    _sample_range(net, diff.sampler_config(True), x, labc, None, k - 1, 1, pred)
    _sample_range(net, diff.sampler_config(True, solver="dpmpp_2m"), x, labc, None, k - 2, k - 1, pred)
    res["m2_first_step_ddim_equal"] = torch.equal(got, x.cpu())
    ddim_k = diff.p_sample(net, shape, noise=x_k, label=label, device="cuda", use_ddim=True, start_step=k)
    res["m2_differs_from_ddim"] = (got - ddim_k).abs().max().item()
    # (6) chunking: several chunks over two lanes and a ragged last chunk (7 images, 2 per chunk under CFG) vs one chunk
    chunked = _model(cfg, ucase["seed"], max_rows=4)
    cinv = diff.ddim_invert(chunked, x0, label=label)
    res["chunked_max_abs"] = (cinv - full).abs().max().item()
    res["chunked_rel"] = res["chunked_max_abs"] / full.abs().max().item()
    res["chunked_equal"] = torch.equal(cinv, full)
    csmp = diff.p_sample(chunked, shape, noise=x_k, label=label, device="cuda", use_ddim=True, start_step=k)
    res["chunked_sample_max_abs"] = (csmp - ddim_k).abs().max().item()
    res["latent_max"] = full.abs().max().item()
    res["finite"] = bool(torch.isfinite(full).all() and torch.isfinite(other).all() and torch.isfinite(got).all())
    return res


def main():
    torch.cuda.set_device(0)
    mode = sys.argv[1]
    if mode == "parity":
        out = parity(sys.argv[2], int(sys.argv[3]), sys.argv[4])
    elif mode == "exactness":
        out = exactness()
    else:
        raise SystemExit(f"unknown mode {mode}")
    print("RESULT " + json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
