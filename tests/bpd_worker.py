"""Child process of tests/test_bpd_gpu.py: one whole-network likelihood case on cuda:0.  Prints one JSON line.

    python -m tests.bpd_worker parity ddim_cfg_v 10 fp16
    python -m tests.bpd_worker exactness
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
from tests.bpd_ref import calc_all_bpd as ref_bpd                                      # noqa: E402
from tests.cases import UNET_CASES, SAMPLE_CASES, build_sample_inputs                  # noqa: E402
from tests.dpm_solver_worker import _diffusion, _model                                 # noqa: E402
from v_diffusion_b200 import _lib                                                      # noqa: E402


def _images(noise):
    """Images on the 8-bit grid of model space, from the case's noise."""
    return torch.round((torch.tanh(noise) + 1) * 127.5) / 127.5 - 1


def _rel(a, b):
    return ((a - b).abs() / b.abs().clamp(min=1e-12)).max().item()


def parity(name, T, operand):
    """Fused and generic calc_all_bpd against the reference bound over the oracle UNet, with the same injected noise."""
    case = SAMPLE_CASES[name]
    ucase = UNET_CASES[case["unet"]]
    cfg = ucase["cfg"]
    noise, label, _ = build_sample_inputs(case, cfg)
    x0 = _images(noise)
    eps = torch.randn((T,) + tuple(x0.shape), generator=torch.Generator().manual_seed(17))
    sd = make_state_dict(cfg, ucase["seed"])
    oracle_net = lambda x, t, y: unet_forward(sd, cfg, x, t, y)                         # noqa: E731
    net = _model(cfg, ucase["seed"], operand)
    diff = _diffusion(case, T)
    ref = ref_bpd(oracle_net, x0, label, eps, T=T, model_out_type=case["model_out_type"], var_type=case["var_type"],
                  intp_frac=case.get("intp_frac"))
    fused = diff.calc_all_bpd(net, x0, y=label, noise=eps)
    generic = diff.calc_all_bpd(lambda x, t, y: net(x, t, y), x0, y=label, noise=eps)
    out = dict(total_ref=ref[0].tolist(), prior_ref=ref[2].tolist())
    for tag, got in (("fused", fused), ("generic", generic)):
        out[tag + "_total_rel"] = _rel(got[0], ref[0])
        out[tag + "_terms_max_abs"] = (got[1] - ref[1]).abs().max().item()
        out[tag + "_terms_rel"] = (got[1] - ref[1]).abs().max().item() / ref[1].abs().max().item()
        out[tag + "_mse_rel"] = (got[3] - ref[3]).abs().max().item() / ref[3].abs().max().item()
        out[tag + "_prior_rel"] = _rel(got[2], ref[2])
    out["fused_vs_generic_rel"] = _rel(fused[0], generic[0])
    out["finite"] = bool(all(torch.isfinite(v).all() for v in fused + generic))
    return out


def _range(net, sc, x0, label, first, num, terms, mse):
    plan = net.plan_for(x0.shape[2], torch.device("cuda", 0))
    _lib.check(_lib.lib().vdt_calc_bpd_range(plan, C.byref(sc), _lib.ptr(x0), _lib.ptr(label), None, 1, x0.shape[0], first, num,
                                             _lib.ptr(terms), _lib.ptr(mse), _lib.current_stream_ptr()))
    torch.cuda.synchronize()


def exactness():
    """Bit-identical properties of the fused evaluation on small_cond (v, labels), on-device noise."""
    case = SAMPLE_CASES["ddim_cfg_v"]
    ucase = UNET_CASES[case["unet"]]
    cfg = ucase["cfg"]
    T, k, B = 12, 5, 7
    diff = _diffusion(case, T)
    g = torch.Generator().manual_seed(43)
    shape = (B, 3, 16, 16)
    x0 = _images(torch.randn(shape, generator=g))
    label = torch.randint(0, 11, (B,), generator=g)
    res = {}
    net = _model(cfg, ucase["seed"])
    full = diff.calc_all_bpd(net, x0, y=label, seed=5)
    # (1) [0, k) then [k, T) == [0, T)
    sc = diff.sampler_config(False, seed=5)
    xd, ld = x0.cuda().contiguous(), label.cuda()
    terms = torch.full((B, T), float("nan"), dtype=torch.float64, device="cuda")
    mse = torch.full_like(terms, float("nan"))
    _range(net, sc, xd, ld, 0, k, terms, mse)
    _range(net, sc, xd, ld, k, T - k, terms, mse)
    res["split_equal"] = torch.equal(terms.cpu(), full[1]) and torch.equal(mse.cpu(), full[3])
    # (2) chunking: several chunks over two lanes and a ragged last chunk (7 images, 3 per chunk) vs one chunk
    chunked = diff.calc_all_bpd(_model(cfg, ucase["seed"], max_rows=3), x0, y=label, seed=5)
    res["chunked_equal"] = all(torch.equal(a, b) for a, b in zip(chunked, full))
    # (3) the same seed repeats, another seed differs
    again = diff.calc_all_bpd(net, x0, y=label, seed=5)
    other = diff.calc_all_bpd(net, x0, y=label, seed=6)
    res["same_seed_equal"] = all(torch.equal(a, b) for a, b in zip(again, full))
    res["other_seed_differs"] = not torch.equal(other[1], full[1])
    res["other_seed_total_diff"] = (other[0] - full[0]).abs().max().item()
    # (4) sampling after a likelihood call on the same plan == sampling on a fresh plan
    noise = torch.randn(shape, generator=g)
    for kw in (dict(use_ddim=True), dict(use_ddim=False, seed=9)):
        a = diff.p_sample(net, shape, noise=noise, label=label, device="cuda", **kw)
        b = diff.p_sample(_model(cfg, ucase["seed"]), shape, noise=noise, label=label, device="cuda", **kw)
        res.setdefault("sample_after_bpd_equal", []).append(torch.equal(a, b))
    res["finite"] = bool(all(torch.isfinite(v).all() for v in full))
    res["total"] = full[0].tolist()
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
