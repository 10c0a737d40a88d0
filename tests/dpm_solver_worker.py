"""Child process of tests/test_dpm_solver_gpu.py: one whole-network DPM-Solver++(2M) case on cuda:0.  Prints one JSON line.

    python -m tests.dpm_solver_worker parity ddim_cfg_v 12 fp16
    python -m tests.dpm_solver_worker progressive ddim_cfg_v 20 fp16x3
    python -m tests.dpm_solver_worker exactness
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
from tests.dpm_solver_ref import p_sample as oracle_p_sample                          # noqa: E402
from tests.cases import UNET_CASES, SAMPLE_CASES, build_sample_inputs                  # noqa: E402
from v_diffusion_b200 import UNet, GaussianDiffusion, get_logsnr_schedule, _lib         # noqa: E402

SOLVER = "dpmpp_2m"


def _model(cfg, seed, operand="fp16", max_rows=None):
    net = UNet(cfg["in_channels"], cfg["hid_channels"], cfg["out_channels"], cfg["ch_multipliers"],
               cfg["num_res_blocks"], cfg["apply_attn"], embedding_dim=cfg["embedding_dim"], head_dim=cfg["head_dim"],
               num_heads=cfg["num_heads"], num_classes=cfg["num_classes"], multitags=cfg["multitags"])
    net.load_state_dict(make_state_dict(cfg, seed), strict=True)
    net.operand_dtype = operand
    if max_rows is not None:
        net.max_rows = max_rows
    return net.cuda().eval()


def _diffusion(case, T):
    return GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), T, case["model_out_type"], case["var_type"],
                             "snr_trunc", "mse", intp_frac=case.get("intp_frac"), w_guide=case["w_guide"])


def _setup(name, T, operand):
    case = SAMPLE_CASES[name]
    ucase = UNET_CASES[case["unet"]]
    cfg = ucase["cfg"]
    noise, label, _ = build_sample_inputs(case, cfg)
    sd = make_state_dict(cfg, ucase["seed"])
    oracle_net = lambda x, t, y: unet_forward(sd, cfg, x, t, y)                         # noqa: E731
    return case, ucase, cfg, noise, label, oracle_net, _model(cfg, ucase["seed"], operand), _diffusion(case, T)


def parity(name, T, operand):
    """Fused and generic-callable 2M sampling against the oracle's 2M loop over the oracle UNet."""
    case, ucase, cfg, noise, label, oracle_net, net, diff = _setup(name, T, operand)
    shape = tuple(noise.shape)
    rec_ref = []
    ref = oracle_p_sample(oracle_net, shape, noise, label, T=T, model_out_type=case["model_out_type"], w_guide=case["w_guide"],
                          use_ddim=True, record=rec_ref, solver=SOLVER)
    ref_ddim = oracle_p_sample(oracle_net, shape, noise, label, T=T, model_out_type=case["model_out_type"],
                               w_guide=case["w_guide"], use_ddim=True)
    fused = diff.p_sample(net, shape, noise=noise, label=label, device="cuda", use_ddim=True, solver=SOLVER)
    rec = []

    def wrapped(x, t, y):
        o = net(x, t, y)
        rec.append(o.cpu())
        return o
    generic = diff.p_sample(wrapped, shape, noise=noise, label=label, device="cuda", use_ddim=True, solver=SOLVER)
    step_rel = [((o - r).norm() / r.norm()).item() for o, (_, r) in zip(rec, rec_ref)]
    return dict(fused_max_abs=(fused - ref).abs().max().item(), generic_max_abs=(generic - ref).abs().max().item(),
                fused_vs_generic=(fused - generic).abs().max().item(), steps=len(rec), worst_step_rel=max(step_rel),
                solver_vs_ddim=(ref - ref_ddim).abs().max().item(), finite=bool(torch.isfinite(fused).all()))


def progressive(name, T, operand):
    """p_sample_progressive(solver="dpmpp_2m") -- several range calls sharing one pred buffer -- against the oracle's
    progressive loop (fp32 step tensor)."""
    case, ucase, cfg, noise, label, oracle_net, net, diff = _setup(name, T, operand)
    shape = tuple(noise.shape)
    pred_freq = 3
    preds_ref = []
    ref = oracle_p_sample(oracle_net, shape, noise, label, T=T, model_out_type=case["model_out_type"], w_guide=case["w_guide"],
                          use_ddim=True, pred_record=preds_ref, t_fp32=True, solver=SOLVER)
    x, preds = diff.p_sample_progressive(net, shape, noise=noise, label=label, device="cuda", use_ddim=True,
                                         pred_freq=pred_freq, solver=SOLVER)
    want = torch.stack([p for ti, p in preds_ref if (ti + 1) % pred_freq == 0][::-1][:T // pred_freq])
    return dict(final_max_abs=(x - ref).abs().max().item(), previews_max_abs=(preds - want).abs().max().item(),
                previews=int(preds.shape[0]), w_guide=case["w_guide"])


def _range(net, sc, x, label, first, num, pred):
    plan = net.plan_for(x.shape[2], torch.device("cuda", 0))
    _lib.check(_lib.lib().vdt_p_sample_range(plan, C.byref(sc), _lib.ptr(x), _lib.ptr(label), None, x.shape[0], first, num,
                                             _lib.ptr(pred), _lib.current_stream_ptr()))
    torch.cuda.synchronize()


def exactness():
    """Bit-identical properties of the fused solver on small_cond with CFG (w = 1, v-prediction)."""
    case = SAMPLE_CASES["ddim_cfg_v"]
    ucase = UNET_CASES[case["unet"]]
    cfg = ucase["cfg"]
    T = 12
    diff = _diffusion(case, T)
    g = torch.Generator().manual_seed(31)
    B = 7
    noise = torch.randn(B, 3, 16, 16, generator=g)
    noise2 = torch.randn(B, 3, 16, 16, generator=g)
    label = torch.randint(0, 11, (B,), generator=g)
    shape = tuple(noise.shape)
    res = {}
    net = _model(cfg, ucase["seed"])
    labc = label.cuda()
    # (1) the solver's first step is DDIM's: one range call from T-1, for x and for the guided x0
    outs = []
    for solver in (None, SOLVER):
        x, pred = noise.cuda().clone(), torch.full_like(noise.cuda(), float("nan"))
        _range(net, diff.sampler_config(True, solver=solver), x, labc, T - 1, 1, pred)
        outs.append((x.cpu(), pred.cpu()))
    res["first_step_equal"] = torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    # (2) T = 1 is DDIM (one step returning the guided x0)
    d1 = _diffusion(case, 1)
    res["t1_equal"] = torch.equal(d1.p_sample(net, shape, noise=noise, label=label, device="cuda", use_ddim=True),
                                  d1.p_sample(net, shape, noise=noise, label=label, device="cuda", use_ddim=True, solver=SOLVER))
    # (3) one full-range call == the same trajectory split into range calls that carry pred_x0 (stale NaNs in the exec's
    #     own pred buffer in between: a range call must take the history from pred_x0)
    full = diff.p_sample(net, shape, noise=noise, label=label, device="cuda", use_ddim=True, solver=SOLVER)
    sc = diff.sampler_config(True, solver=SOLVER)
    x, pred = noise.cuda().clone(), torch.empty_like(noise.cuda())
    first = T - 1
    for n in (1, 4, 2, 3, 2):
        _range(net, sc, x, labc, first, n, pred)
        junk = torch.full_like(x, float("nan"))                 # a first step on the same exec leaves NaN in its pred buffer
        _range(net, sc, junk, labc, T - 1, 1, None)
        first -= n
    assert first == -1
    res["split_equal"] = torch.equal(x.cpu(), full)
    res["split_max_abs"] = (x.cpu() - full).abs().max().item()
    # (4) several chunks over two lanes and a ragged last chunk (7 images, 2 per chunk under CFG) vs one chunk
    chunked = _model(cfg, ucase["seed"], max_rows=4)
    c2m = diff.p_sample(chunked, shape, noise=noise, label=label, device="cuda", use_ddim=True, solver=SOLVER)
    cdd = diff.p_sample(chunked, shape, noise=noise, label=label, device="cuda", use_ddim=True)
    fdd = diff.p_sample(net, shape, noise=noise, label=label, device="cuda", use_ddim=True)
    res["chunked_max_abs"] = (c2m - full).abs().max().item()
    res["chunked_equal"] = torch.equal(c2m, full)
    res["ddim_chunked_equal"] = torch.equal(cdd, fdd)                     # the same property of the existing sampler
    # (5) a cached exec called again with other noise gives fresh results: equal to a fresh plan's, and the first input
    #     again reproduces the first output
    other = diff.p_sample(net, shape, noise=noise2, label=label, device="cuda", use_ddim=True, solver=SOLVER)
    fresh = diff.p_sample(_model(cfg, ucase["seed"]), shape, noise=noise2, label=label, device="cuda", use_ddim=True,
                          solver=SOLVER)
    again = diff.p_sample(net, shape, noise=noise, label=label, device="cuda", use_ddim=True, solver=SOLVER)
    res["repeat_fresh_equal"] = torch.equal(other, fresh) and torch.equal(again, full)
    res["differs_from_ddim"] = (full - fdd).abs().max().item()
    res["finite"] = bool(torch.isfinite(full).all() and torch.isfinite(other).all())
    return res


def main():
    torch.cuda.set_device(0)
    mode = sys.argv[1]
    if mode == "parity":
        out = parity(sys.argv[2], int(sys.argv[3]), sys.argv[4])
    elif mode == "progressive":
        out = progressive(sys.argv[2], int(sys.argv[3]), sys.argv[4])
    elif mode == "exactness":
        out = exactness()
    else:
        raise SystemExit(f"unknown mode {mode}")
    print("RESULT " + json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
