"""CPU dry run of tests/train_step_worker.py (the GPU test's child process) with stand-ins for everything that needs a device:
ContractOps for the kernels, an autograd train_loss, a torch AdamW/EMA for the optimizer kernel, .cuda() as identity.  It checks
nothing about the kernels -- it exists so that a typo in the worker or in TrainingStep's host logic is found here and not on
the one hardware run the GPU suite gets.  Usage: python scripts/dryrun_train_worker.py"""
import math
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch.distributed  # noqa: F401,E402  (before the patches below: its import reads torch.Generator as a type)
import torch.optim  # noqa: F401,E402

torch.Tensor.cuda = lambda self, *a, **k: self
torch.nn.Module.cuda = lambda self, *a, **k: self
torch.cuda.synchronize = lambda *a, **k: None
torch.cuda.set_device = lambda *a, **k: None
_Gen = torch.Generator


class _CpuGen(_Gen):                                                        # "cuda" generators -> CPU
    def __new__(cls, device="cpu"):
        return _Gen()


torch.Generator = _CpuGen
_rand, _empty = torch.rand, torch.empty
torch.rand = lambda *a, **k: _rand(*a, **{kk: v for kk, v in k.items() if kk != "device"})
torch.empty = lambda *a, **k: _empty(*a, **{kk: v for kk, v in k.items() if kk != "device"})

from oracle import train_loss as oracle_train_loss                        # noqa: E402
from tests.test_training_graph import ContractOps                         # noqa: E402
import v_diffusion_b200.training as T                                     # noqa: E402
import v_diffusion_b200.optim as O                                        # noqa: E402
from v_diffusion_b200 import GaussianDiffusion, _lib                      # noqa: E402


class Ops32(ContractOps):
    dt = torch.float32
    acc = torch.float32

    @staticmethod
    def _mask(shape, drop_p, seed, layer):
        m = ContractOps._mask(shape, drop_p, seed, layer)
        return None if m is None else m.float()


T.KernelOps = lambda operand="fp16": Ops32()


def fake_train_loss(self, denoise_fn, x_0, t, y, noise=None, return_grad=False):
    hold = {}

    def fn(a, b, c):
        hold["o"] = denoise_fn(a, b, c).detach().requires_grad_(True)
        return hold["o"]
    with torch.enable_grad():
        per, _ = oracle_train_loss(fn, x_0, t, y, noise, model_out_type=self.model_out_type, reweight_type=self.reweight_type)
        per.mean().backward()
    return (per.detach(), hold["o"].grad) if return_grad else per.detach()


GaussianDiffusion.train_loss = fake_train_loss


class FakeAdamWEMA:
    def __init__(self, named_params, lr=2e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, grad_norm=1.0, ema_decay=0.9999, use_ema=True):
        self.params = dict(named_params)
        self.opt = torch.optim.AdamW(list(self.params.values()), lr=lr, betas=betas, eps=eps, weight_decay=weight_decay)
        self.grad_norm, self.decay, self.n = grad_norm, ema_decay, 0
        self.shadow = {k: p.detach().clone() for k, p in self.params.items()} if use_ema else {}

    def step(self, grads, lr=None):
        for k, p in self.params.items():
            p.grad = grads[k].clone()
        total = torch.nn.utils.clip_grad_norm_(list(self.params.values()), max_norm=self.grad_norm)
        self.opt.step()
        self.n += 1
        d = min(self.decay, (1 + self.n) / (10 + self.n))
        with torch.no_grad():
            for k in self.shadow:
                self.shadow[k] += (1 - d) * (self.params[k] - self.shadow[k])
        return (total.double() ** 2).reshape(1)


O.AdamWEMA = FakeAdamWEMA
_dev = torch.device
T.TrainingStep.__init__.__defaults__                                        # (signature untouched)
import tests.train_step_worker as W                                       # noqa: E402

_orig_init = T.TrainingStep.__init__


def _init(self, model, diffusion, **kw):
    kw["device"] = "cuda"                                                   # passes the "CUDA only" gate; tensors stay on the CPU
    _orig_init(self, model, diffusion, **kw)
    self.device = _dev("cpu")


T.TrainingStep.__init__ = _init
W.TrainingStep = T.TrainingStep
_lib.lib().vdt_kernel_launches.restype = __import__("ctypes").c_uint64

if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "ddp":
    # one rank of tests/train_step_ddp_worker.py (the two-GPU NCCL case) on the CPU over gloo; RANK / WORLD_SIZE / MASTER_* from the env
    import torch.distributed as dist
    _init_pg = dist.init_process_group
    dist.init_process_group = lambda backend=None, **kw: _init_pg("gloo", **kw)
    import tests.train_step_ddp_worker as D
    D.TrainingStep = T.TrainingStep
    D.main()
    sys.exit(0)

if __name__ == "__main__":
    r = W.graph_parity("small", 2, "fp16")
    print("graph_parity", {k: r[k] for k in ("out_rel", "grad_rel_worst", "grad_rel_median", "finite")})
    assert r["finite"] and r["out_rel"] < 1e-5 and r["grad_rel_worst"] < 1e-3, r
    r = W.dropout("small", 2, "fp16")
    print("dropout", r)
    assert r["reproducible"] and r["finite"] and r["seed_changes_output"] > 1e-2 and r["eval_differs"] > 1e-2 and r["out_bias_grad_rel"] < 1e-5
    r = W.train_steps("small", 2, "fp16", steps=2)
    print("train_steps", {k: v for k, v in r.items()})
    assert r["loss_rel_worst"] < 1e-5 and r["gnorm_rel_worst"] < 1e-4 and r["cosine_of_updates"] > 0.999 and r["ema_rel_worst"] < 1e-5, r
    r = W.grad_golden("small", 0, "fp16")
    print("grad_golden", {k: r[k] for k in ("loss_rel", "norm_rel_worst", "proj_err_worst", "full_rel_worst", "n_params", "n_full")})
    assert r["loss_rel"] < 1e-5 and r["norm_rel_worst"] < 1e-4 and r["proj_err_worst"] < 1e-3 and r["full_rel_worst"] < 1e-4, r
    from v_diffusion_b200 import UNet as _U
    _U._forward_plan = lambda self, x, t, y=None: torch.zeros(x.shape[0], self.out_channels, x.shape[2], x.shape[3])   # plan path needs a GPU
    r = W.autograd_step("small", 0, "fp16")
    print("autograd_step", {k: r[k] for k in ("loss_rel", "norm_rel_worst", "proj_err_worst", "full_rel_worst", "plan_path_finite")})
    assert r["loss_rel"] < 1e-5 and r["norm_rel_worst"] < 1e-4 and r["proj_err_worst"] < 1e-3 and r["full_rel_worst"] < 1e-4, r
    # bench.py's BASELINE configs[4] block (child process body), tiny batch, CPU stand-ins
    import time
    import bench

    class _Ev:
        def __init__(self, enable_timing=True):
            self.t = None

        def record(self):
            self.t = time.perf_counter()

        def elapsed_time(self, other):
            return (other.t - self.t) * 1e3
    torch.cuda.Event = _Ev
    torch.cuda.empty_cache = lambda: None
    bench.CIFAR_COND_MODEL = dict(bench.CIFAR_COND_MODEL, hid_channels=64, num_res_blocks=1)     # keep the dry run short
    bench.stage_cfg = None
    from oracle import stage_ref
    _cfg0 = stage_ref.config

    def _small(name):
        c = _cfg0(name)
        c["model"] = dict(c["model"], hid_channels=64, num_res_blocks=1)
        return c
    stage_ref.config = _small
    bench.train_step_child(batch=2, steps=1, device=_dev("cpu"))
    print("dry run OK")
