"""GPU: DPM-Solver++(2M) sampling (solver="dpmpp_2m").  The fused update kernel against the fp64 step formula, the closed-form
Gaussian case through the generic path against the oracle, whole small networks against the oracle's 2M loop (each in a child
process, tests/dpm_solver_worker.py), the bit-identical properties of the fused solver, and the generate driver.  Bars are the
sampler's existing ones (tests/test_gpu_unet.py)."""
import json
import os
import subprocess
import sys
import zlib

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REL_L2 = 1e-2
SAMPLE_MAX_ABS = 2e-2
VALIDATION_MAX_ABS = 1e-3


def _run(*args, timeout=1800):
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run([sys.executable, "-m", "tests.dpm_solver_worker", *map(str, args)], cwd=ROOT, env=env, capture_output=True,
                       text=True, timeout=timeout)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")]
    assert r.returncode == 0 and lines, (r.stdout[-1500:] + "\n" + r.stderr[-2500:])
    res = json.loads(lines[-1][len("RESULT "):])
    print(" ".join(map(str, args)), "->", json.dumps(res))
    return res


def _step_fp64(out_type, model_out, x, coef, cfg, w, pred_prev):
    """One guided 2M step in fp64 from the fp32 coefficient row (include/vdt_b200.h slot layout)."""
    cf = coef.double()
    x = x.double()

    def x0(o):
        if out_type == 3:
            v = x * cf[0] - o * cf[1]
        elif out_type == 0:
            v = o
        elif out_type == 1:
            v = x * cf[2] - o * cf[3]
        else:
            xo, eo = o.chunk(2, dim=1)
            v = xo * cf[5] + (x * cf[2] - eo * cf[3]) * cf[4]
        return v.clamp(-1, 1)
    mo = model_out.double()
    if cfg:
        x0c, x0u = x0(mo[0::2]), x0(mo[1::2])
        mean_c, mean_u = cf[6] * x + cf[7] * x0c, cf[6] * x + cf[7] * x0u
        mean, pred = mean_c + w * (mean_c - mean_u), x0c + w * (x0c - x0u)
    else:
        pred = x0(mo)
        mean = cf[6] * x + cf[7] * pred
    if cf[15] != 0:
        mean = mean + cf[15] * (pred - pred_prev.double())
    return mean, pred


@pytest.mark.parametrize("out_type", ["x0", "eps", "both", "v"])
@pytest.mark.parametrize("cfg", [False, True])
@pytest.mark.parametrize("hw", [(16, 16), (5, 7)])                    # 5 x 7: odd C*H*W, the scalar (VEC = 1) kernel
def test_sampler_step_hist_kernel_vs_fp64(out_type, cfg, hw):
    from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule, _lib
    L = _lib.lib()
    T, ti, B, Cc = 20, 9, 3, 3
    d = GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), T, out_type, "fixed_large", "snr_trunc", "mse", w_guide=1.5)
    coefs = d.step_coefficients(True, solver="dpmpp_2m")
    assert coefs[ti, 15] != 0
    g = torch.Generator().manual_seed(zlib.crc32(f"{out_type}{cfg}{hw}".encode()))
    H, W = hw
    Cm = 2 * Cc if out_type == "both" else Cc
    x = torch.randn(B, Cc, H, W, generator=g)
    mo = torch.randn(B * (2 if cfg else 1), Cm, H, W, generator=g) * 0.6
    prev = torch.rand(B, Cc, H, W, generator=g) * 2 - 1
    want_x, want_pred = _step_fp64(_lib.OUT_TYPES[out_type], mo, x, coefs[ti], cfg, 1.5, prev)
    xs = torch.empty(B, Cc, H, W, device="cuda")
    hist = prev.cuda()
    mo_d, x_d = mo.cuda(), x.cuda()                    # held for the whole test: the library only sees their addresses
    _lib.check(L.vdt_op_sampler_step_hist(_lib.ptr(mo_d), _lib.ptr(x_d), None, _lib.ptr(xs), B, Cc, H * W, int(cfg),
                                          _lib.OUT_TYPES[out_type], ti, _lib.ptr(coefs[ti].contiguous()), 1.5, _lib.ptr(hist),
                                          _lib.current_stream_ptr()))
    rel_x = ((xs.cpu().double() - want_x).abs().max() / want_x.abs().max()).item()
    rel_p = ((hist.cpu().double() - want_pred).abs().max() / want_pred.abs().max()).item()
    print(f"{out_type} cfg={cfg} {hw}: x_s {rel_x:.2e} pred {rel_p:.2e}")
    assert rel_x <= 1e-6 and rel_p <= 1e-6
    # a first-order row (c2k = 0) never reads the history: NaNs there change nothing, bit for bit against the old entry point
    ddim = d.step_coefficients(True)[ti].contiguous()
    a, b = torch.empty_like(xs), torch.empty_like(xs)
    nan_hist = torch.full_like(xs, float("nan"))
    args = (_lib.ptr(mo_d), _lib.ptr(x_d), None)
    _lib.check(L.vdt_op_sampler_step(*args, _lib.ptr(a), B, Cc, H * W, int(cfg), _lib.OUT_TYPES[out_type], ti, _lib.ptr(ddim), 1.5,
                                     _lib.current_stream_ptr()))
    _lib.check(L.vdt_op_sampler_step_hist(*args, _lib.ptr(b), B, Cc, H * W, int(cfg), _lib.OUT_TYPES[out_type], ti, _lib.ptr(ddim),
                                          1.5, _lib.ptr(nan_hist), _lib.current_stream_ptr()))
    assert torch.equal(a, b) and torch.isfinite(nan_hist).all()
    # the history-less entry point refuses a 2M row
    assert L.vdt_op_sampler_step(*args, _lib.ptr(a), B, Cc, H * W, int(cfg), _lib.OUT_TYPES[out_type], ti,
                                 _lib.ptr(coefs[ti].contiguous()), 1.5, _lib.current_stream_ptr()) != 0
    assert "vdt_op_sampler_step_hist" in L.vdt_last_error().decode()


def test_closed_form_case_through_the_generic_path():
    """The Gaussian closed-form denoiser of tests/test_dpm_solver_cpu.py as a generic callable on the GPU: the same 2M
    trajectory as the oracle's to fp32 rounding."""
    from tests.dpm_solver_ref import p_sample as oracle_p_sample
    from tests.test_dpm_solver_cpu import _posterior_mean
    from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule
    xT = 0.75 * torch.randn(2, 3, 8, 8, generator=torch.Generator().manual_seed(0))
    for T in (10, 40):
        d = GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), T, "x0", "fixed_large", "snr_trunc", "mse", w_guide=0.0)
        got = d.p_sample(lambda x, t, y: _posterior_mean(x.cpu(), t.cpu()).cuda(), tuple(xT.shape), noise=xT, device="cuda",
                         use_ddim=True, solver="dpmpp_2m")
        ref = oracle_p_sample(_posterior_mean, tuple(xT.shape), xT, None, T=T, model_out_type="x0", use_ddim=True,
                              solver="dpmpp_2m")
        err = (got - ref).abs().max().item()
        print(f"closed form T={T}: GPU generic path vs oracle {err:.2e}")
        assert err <= 1e-5


@pytest.mark.parametrize("name,T", [("ddim_cfg_v", 12), ("ddim_x0_uncond", 10), ("ddim_cfg_multitag", 8)])
@pytest.mark.parametrize("operand", ["fp16", "fp16x3"])
def test_unet_sampling_vs_oracle(name, T, operand):
    """small_cond (CFG w = 1, v), small_hd64_x0 (unconditional, x0) and small_multitag (CFG w = 1, multi-hot labels): fused
    and generic 2M sampling against the oracle's 2M loop over the oracle UNet."""
    res = _run("parity", name, T, operand)
    bar = SAMPLE_MAX_ABS if operand == "fp16" else VALIDATION_MAX_ABS
    assert res["finite"] and res["steps"] == T
    assert res["fused_max_abs"] <= bar and res["generic_max_abs"] <= bar, res
    assert res["worst_step_rel"] <= REL_L2, res
    assert res["fused_vs_generic"] <= 1e-5, res
    assert res["solver_vs_ddim"] > 1e-3, res                   # the solver changes the trajectory


@pytest.mark.parametrize("operand", ["fp16", "fp16x3"])
def test_progressive_vs_oracle(operand):
    res = _run("progressive", "ddim_cfg_v", 20, operand)
    bar = SAMPLE_MAX_ABS if operand == "fp16" else VALIDATION_MAX_ABS
    assert res["previews"] == 6
    assert res["final_max_abs"] <= bar, res
    assert res["previews_max_abs"] <= bar * (1.0 + res["w_guide"]), res


def test_fused_solver_exactness_properties():
    res = _run("exactness")
    assert res["finite"]
    assert res["first_step_equal"], res                     # the first step is DDIM's
    assert res["t1_equal"], res                             # T = 1 is DDIM
    assert res["split_equal"], res                          # range calls carrying pred_x0 == one call
    assert res["repeat_fresh_equal"], res                   # a cached exec never reads stale history
    # chunking: the same bar as the existing sampler's chunking property (conv tiles depend on the chunk's image count);
    # bit-identical whenever DDIM itself is
    assert res["chunked_max_abs"] <= 1e-5, res
    assert res["chunked_equal"] or not res["ddim_chunked_equal"], res
    assert res["differs_from_ddim"] > 1e-3, res


def test_generate_driver_with_solver(tmp_path):
    """`python -m v_diffusion_b200.generate --use-ddim --solver dpmpp_2m` equals p_sample(solver="dpmpp_2m") on the driver's
    seeded noise and labels."""
    from oracle.unet_ref import make_state_dict
    from tests.cases import UNET_CASES
    from tests.dpm_solver_worker import _model
    from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule
    from v_diffusion_b200.generate import images_to_uint8
    ucase = UNET_CASES["small_cond"]
    cfg = ucase["cfg"]
    torch.save({"model": make_state_dict(cfg, ucase["seed"])}, tmp_path / "ckpt.pt")
    merged = json.load(open(os.path.join(ROOT, "tests", "golden", "merged_configs.json")))["cifar10_cond"]
    model_block = dict(in_channels=3, hid_channels=64, ch_multipliers=[1, 2], num_res_blocks=2, apply_attn=[False, True],
                       drop_rate=0.2, num_heads=1)
    json.dump({"data": {"name": "cifar10"}, "model": model_block, "diffusion": merged["diffusion"],
               "conditional": merged["conditional"]}, open(tmp_path / "cfg.json", "w"))
    json.dump({}, open(tmp_path / "defaults.json", "w"))
    total, bs, T, seed = 6, 4, 10, 5
    cmd = [sys.executable, "-m", "v_diffusion_b200.generate", "--config-path", str(tmp_path / "cfg.json"), "--default-config-path",
           str(tmp_path / "defaults.json"), "--ckpt-path", str(tmp_path / "ckpt.pt"), "--sample-timesteps", str(T), "--w-guide", "1.0",
           "--batch-size", str(bs), "--total-size", str(total), "--save-path", str(tmp_path / "out.pt"), "--seed", str(seed),
           "--use-ddim", "--solver", "dpmpp_2m"]
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    got = torch.load(tmp_path / "out.pt")
    net = _model(cfg, ucase["seed"])
    d = merged["diffusion"]
    diff = GaussianDiffusion(get_logsnr_schedule(d["logsnr_schedule"], d["logsnr_min"], d["logsnr_max"]), T, d["model_out_type"],
                             d["model_var_type"], d["reweight_type"], d["loss_type"], intp_frac=d["intp_frac"], w_guide=1.0)
    gen = torch.Generator(device="cuda").manual_seed(seed)
    want, ddim = [], []
    for b0 in range(0, total, bs):
        n = min(bs, total - b0)
        noise = torch.randn((n, 3, 32, 32), device="cuda", generator=gen)
        label = torch.randint(10, (n,), device="cuda", generator=gen) + 1
        call_seed = int(torch.randint(0, 2 ** 62, (1,), device="cuda", generator=gen).item())
        want.append(diff.p_sample(net, (n, 3, 32, 32), noise=noise, label=label, device="cuda", seed=call_seed, use_ddim=True,
                                  solver="dpmpp_2m"))
        ddim.append(diff.p_sample(net, (n, 3, 32, 32), noise=noise, label=label, device="cuda", seed=call_seed, use_ddim=True))
    want = images_to_uint8(torch.cat(want).cuda()).cpu()
    assert torch.equal(got, want)
    assert not torch.equal(got, images_to_uint8(torch.cat(ddim).cuda()).cpu())
