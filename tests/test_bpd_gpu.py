"""GPU: the likelihood bound in bits/dim.  The term kernel against the fp64 step formula, the closed-form pin through the generic
path, whole small networks against the reference bound over the oracle UNet (each in a child process, tests/bpd_worker.py),
the bit-identical properties of the fused path, and the command line.  The whole-network bars sit 2-5x above the worst values
measured on a B200 (profiles/r9_bpd_parity.txt)."""
import json
import os
import subprocess
import sys
import zlib

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# total, every term and mse, relative to the reference (worst measured: 1.9e-4 in fp16, 5.8e-7 in fp16x3)
TOTAL_REL = {"fp16": 5e-4, "fp16x3": 2e-6}


def _run(*args, timeout=1800):
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run([sys.executable, "-m", "tests.bpd_worker", *map(str, args)], cwd=ROOT, env=env, capture_output=True,
                       text=True, timeout=timeout)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("RESULT ")]
    assert r.returncode == 0 and lines, (r.stdout[-1500:] + "\n" + r.stderr[-2500:])
    res = json.loads(lines[-1][len("RESULT "):])
    print(" ".join(map(str, args)), "->", json.dumps(res))
    return res


def _offset(t, off):
    """A copy of t whose storage starts `off` elements into a fresh buffer (off = 1: not 16-byte aligned)."""
    buf = torch.empty(t.numel() + off, device="cuda", dtype=t.dtype)
    v = buf[off:].view(t.shape)
    v.copy_(t)
    return v


def _output_for(out_type, x0_hat, x_t, cf):
    """fp32 raw model output whose x0 prediction at the row's converters is x0_hat (fp64 inversion of the converters)."""
    cf, x = cf.double(), x_t.double()
    if out_type == "x0":
        return x0_hat.float()
    if out_type == "eps":
        return ((x * cf[2] - x0_hat) / cf[3]).float()
    if out_type == "v":
        return ((x * cf[0] - x0_hat) / cf[1]).float()
    return torch.cat([x0_hat, (x * cf[2] - x0_hat) / cf[3]], dim=1).float()      # both halves predict x0_hat


@pytest.mark.parametrize("out_type", ["x0", "eps", "both", "v"])
@pytest.mark.parametrize("clip", [True, False])
@pytest.mark.parametrize("hw,off", [((16, 16), 0), ((16, 16), 1), ((5, 7), 0), ((80, 80), 0)])   # odd offset / odd C*H*W: scalar
def test_bpd_term_kernel_vs_fp64(out_type, clip, hw, off):
    """80x80x3 spans several 4096-element tiles.  Step 0 (the decoder, fixed_large so its bins are not a delta) with outputs whose
    x0_hat lies within about a bin of x0, where the fp32 decoder is well conditioned, and two KL steps with outputs whose x0_hat
    falls beyond [-1, 1] (so the clip acts)."""
    from tests.bpd_ref import bpd_coefficients, step_terms
    from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule, _lib
    L = _lib.lib()
    T, B, Cc = 20, 3, 3
    d = GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), T, out_type, "fixed_large", "snr_trunc", "mse")
    coefs = d.bpd_coefficients()
    co = bpd_coefficients(T, "fixed_large")
    g = torch.Generator().manual_seed(zlib.crc32(f"{out_type}{clip}{hw}{off}".encode()))
    H, W = hw
    Cm = 2 * Cc if out_type == "both" else Cc
    terms = _offset(torch.zeros(B, T, dtype=torch.float64, device="cuda"), off)
    mse = _offset(torch.zeros(B, T, dtype=torch.float64, device="cuda"), off)
    for i in (0, 9, T - 1):
        x0 = torch.round((torch.rand(B, Cc, H, W, generator=g) * 2 - 1) * 127.5) / 127.5     # the 8-bit grid, edges included
        x0[:, 0, 0, 0], x0[:, 0, 0, 1] = -1.0, 1.0
        x_t = torch.randn(B, Cc, H, W, generator=g)
        mo = torch.randn(B, Cm, H, W, generator=g) * 1.5
        if i == 0:
            mo = _output_for(out_type, x0.double() + 0.005 * torch.randn(x0.shape, generator=g, dtype=torch.float64), x_t, coefs[0])
        want_t, want_m = step_terms(mo, x_t, x0, i, co, out_type, clip)
        mo_d, xt_d, x0_d = _offset(mo.cuda(), off), _offset(x_t.cuda(), off), _offset(x0.cuda(), off)
        _lib.check(L.vdt_op_bpd_term(_lib.ptr(mo_d), _lib.ptr(xt_d), _lib.ptr(x0_d), B, Cc, H * W, _lib.OUT_TYPES[out_type], i, T,
                                     _lib.ptr(coefs[i].contiguous()), int(clip), _lib.ptr(terms), _lib.ptr(mse),
                                     _lib.current_stream_ptr()))
        got_t, got_m = terms[:, i].cpu(), mse[:, i].cpu()
        rel_m = ((got_m - want_m).abs() / want_m).max().item()
        rel_t = ((got_t - want_t).abs() / want_t.abs()).max().item()
        print(f"{out_type} clip={clip} {hw} off={off} step {i}: mse {rel_m:.2e} term {rel_t:.2e}")
        assert rel_m <= 1e-5, (i, rel_m)
        assert rel_t <= 1e-5, (i, rel_t)


def test_cheating_denoiser_through_the_generic_path():
    """Closed-form pin (a) on the GPU: an x0 model returning the true x0 under fixed_small makes every term with i > 0 exactly 0,
    so the total is the prior plus the decoder; the prior and decoder equal the reference's."""
    from tests.bpd_ref import calc_all_bpd as ref_bpd
    from tests.test_dpm_solver_cpu import S
    from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule
    T = 12
    x0 = (S * torch.randn(3, 3, 8, 8, generator=torch.Generator().manual_seed(0))).clamp(-1, 1)
    noise = torch.randn((T,) + tuple(x0.shape), generator=torch.Generator().manual_seed(1))
    d = GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), T, "x0", "fixed_small", "snr_trunc", "mse")
    xd = x0.cuda()
    total, terms, prior, mse = d.calc_all_bpd(lambda x, t, y: xd, x0, noise=noise)
    assert torch.all(terms[:, 1:] == 0) and torch.all(mse == 0)
    assert torch.equal(total, terms.sum(1) + prior)
    rt, _, rp, _ = ref_bpd(lambda x, t, y: x0, x0, None, noise, T=T, model_out_type="x0", var_type="fixed_small")
    assert torch.allclose(prior, rp, rtol=1e-12, atol=0) and torch.allclose(total, rt, rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("name,T", [("ddim_cfg_v", 10), ("ddim_cfg_multitag", 8), ("ancestral_both", 8)])
@pytest.mark.parametrize("operand", ["fp16", "fp16x3"])
def test_unet_bpd_vs_reference(name, T, operand):
    """small_cond (v, labels, fixed_medium), small_multitag (v, multi-hot labels, fixed_large) and small_hd64 ("both",
    unconditional, fixed_large): fused and generic calc_all_bpd against the reference bound over the oracle UNet."""
    res = _run("parity", name, T, operand)
    assert res["finite"]
    for tag in ("fused", "generic"):
        assert res[tag + "_total_rel"] <= TOTAL_REL[operand], res
        assert res[tag + "_terms_rel"] <= TOTAL_REL[operand] and res[tag + "_mse_rel"] <= TOTAL_REL[operand], res
        assert res[tag + "_prior_rel"] <= 1e-12, res
    assert res["fused_vs_generic_rel"] <= 1e-5, res


def test_fused_exactness_properties():
    res = _run("exactness")
    assert res["finite"]
    assert res["split_equal"], res                          # [0, k) then [k, T) == [0, T)
    assert res["chunked_equal"], res                        # chunks and lanes do not change a bit
    assert res["same_seed_equal"] and res["other_seed_differs"], res
    assert all(res["sample_after_bpd_equal"]), res          # the sampler's execs are untouched


def _cli(tmp_path, nproc):
    out = tmp_path / f"bpd{nproc}.json"
    cmd = ["-m", "v_diffusion_b200.bpd", "--config-path", str(tmp_path / "cfg.json"), "--ckpt-path", str(tmp_path / "ckpt.pt"),
           "--use-ema", "--images", str(tmp_path / "x.npy"), "--labels", str(tmp_path / "y.npy"), "--sample-timesteps", "6",
           "--batch-size", "3", "--seed", "11", "--out", str(out)]
    if nproc > 1:
        cmd = ["-m", "torch.distributed.run", "--standalone", f"--nproc-per-node={nproc}"] + cmd
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run([sys.executable] + cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-3000:]
    return json.load(open(out))


def test_cli_on_a_training_step_checkpoint(tmp_path):
    """`python -m v_diffusion_b200.bpd` on a checkpoint written by TrainingStep (EMA weights), on one GPU and, when present, two:
    both give the same per-image results, equal to calc_all_bpd on the same batches and seeds."""
    import numpy as np
    from oracle.unet_ref import make_state_dict
    from tests.cases import UNET_CASES
    from tests.dpm_solver_worker import _model
    from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule
    from v_diffusion_b200.bpd import images_to_model_space
    from v_diffusion_b200.training import TrainingStep
    ucase = UNET_CASES["small_cond"]
    cfg = ucase["cfg"]
    net = _model(cfg, ucase["seed"])
    diff = GaussianDiffusion(get_logsnr_schedule("cosine", -20., 20.), 6, "v", "fixed_large", "snr_trunc", "mse")
    TrainingStep(net, diff, use_ema=True).save_checkpoint(str(tmp_path / "ckpt.pt"))
    model_block = dict(in_channels=3, hid_channels=64, ch_multipliers=[1, 2], num_res_blocks=2, apply_attn=[False, True],
                       drop_rate=0.0, num_heads=1)
    json.dump({"data": {"name": "cifar10"}, "model": model_block,
               "diffusion": dict(logsnr_schedule="cosine", logsnr_min=-20., logsnr_max=20., allow_rescale=False, train_timesteps=0,
                                 sample_timesteps=6, model_out_type="v", model_var_type="fixed_large", reweight_type="snr_trunc",
                                 loss_type="mse", intp_frac=0.0, x0eps_coef=False)},
              open(tmp_path / "cfg.json", "w"))
    g = np.random.default_rng(0)
    N = 7
    np.save(tmp_path / "x.npy", g.integers(0, 256, size=(N, 32, 32, 3), dtype=np.uint8))
    np.save(tmp_path / "y.npy", g.integers(1, 11, size=(N,)))
    one = _cli(tmp_path, 1)
    assert one["images"] == N and one["sample_timesteps"] == 6 and len(one["terms_bpd_mean"]) == 6
    ref = _model(cfg, ucase["seed"])
    ref.load_state_dict(make_state_dict(cfg, ucase["seed"]))
    x = images_to_model_space(np.load(tmp_path / "x.npy"), "cuda")
    y = torch.from_numpy(np.load(tmp_path / "y.npy"))
    want = torch.cat([diff.calc_all_bpd(ref, x[k:k + 3], y=y[k:k + 3], seed=11 + k // 3)[0] for k in range(0, N, 3)])
    assert one["total_bpd"] == want.tolist()
    if torch.cuda.device_count() >= 2:
        assert _cli(tmp_path, 2)["total_bpd"] == one["total_bpd"]
