"""CPU tests of the composed training step's host logic (v-diffusion-torch_b200/training.py).

The product runs ``UNetTrainGraph`` on ``KernelOps`` (ctypes into the CUDA library, no fallback).  What can be checked
without a GPU is the *orchestration* (the tests monkeypatch the module's ``KernelOps`` name; the package has no backend switch): the block order read off the module tree, which tensor feeds which call, where every
gradient flows (concat splits, the skip stack, resample adjoints, the FiLM / embedding chain, in_conv's im2col and out_conv's
padded GEMM).  ``ContractOps`` below is test infrastructure: it models the documented contract of each kernel-level entry point
(include/vdt_b200.h) with fp64 torch ops, so the graph's output and every parameter gradient can be compared with autograd
through the oracle UNet.  The kernels themselves are checked one by one on the GPU (tests/test_gpu_kernels.py) and the graph on
the real kernels in tests/test_train_step_gpu.py.
"""
import math
import os
import sys

import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import make_state_dict                                       # noqa: E402
from oracle.unet_ref import _unet_forward                                # noqa: E402
from oracle.diffusion_ref import timestep_embedding                      # noqa: E402
from tests.cases import _cfg                                             # noqa: E402
from v_diffusion_b200 import UNet                                        # noqa: E402
from v_diffusion_b200.training import (UNetTrainGraph, GradBucketReducer, block_list, pow2_scale_for_16bit,   # noqa: E402
                                       _resample_adjoint)


class ContractOps:
    """fp64 model of the vdt_op_* contracts (NHWC activations, OIHW weights); gradients by autograd of the same formula."""
    dt = torch.float64
    acc = torch.float64
    f16 = 1

    def __init__(self):
        self.calls = []

    def to16(self, x):
        return x

    def grad16(self, g):
        return g, None

    @staticmethod
    def _rs(z, resample):
        if resample == 1:
            return F.avg_pool2d(z, 2)
        if resample == 2:
            return F.interpolate(z, scale_factor=2, mode="nearest")
        return z

    @staticmethod
    def _mask(shape, drop_p, seed, layer):
        if drop_p <= 0:
            return None
        g = torch.Generator().manual_seed((seed * 1315423911 + layer) % (2 ** 63))
        return (torch.rand(shape, generator=g, dtype=torch.float64) >= drop_p).double() / (1 - drop_p)

    def _gn(self, x, gamma, beta, film, silu, mask):
        Cc = x.shape[3]
        y = F.group_norm(x.permute(0, 3, 1, 2), 32, gamma, beta, 1e-6)
        if film is not None:
            shift, scale = film[:, :Cc, None, None], film[:, Cc:2 * Cc, None, None]
            y = (1 + scale) * y + shift
        if silu:
            y = F.silu(y)
        y = y.permute(0, 2, 3, 1)
        return y if mask is None else y * mask

    def groupnorm(self, src1, src2, gamma, beta, film, silu, resample, want_raw, want_res):
        self.calls.append("groupnorm")
        x = src1 if src2 is None else torch.cat([src1, src2], dim=3)
        act = self._rs(self._gn(x, gamma, beta, film, silu, None).permute(0, 3, 1, 2), resample).permute(0, 2, 3, 1).contiguous()
        raw = x.clone() if want_raw else None
        res = self._rs(x.permute(0, 3, 1, 2), resample).permute(0, 2, 3, 1).contiguous() if want_res else None
        return act, raw, res

    def groupnorm_train(self, src, gamma, beta, film, drop_p, seed, layer):
        self.calls.append("groupnorm_train")
        return self._gn(src, gamma, beta, film, True, self._mask(src.shape, drop_p, seed, layer)).contiguous()

    def conv(self, a16, w, b, residual, ksize, out16=False):
        self.calls.append(f"conv{ksize}")
        assert a16.is_contiguous() and w.shape[1] == a16.shape[3] and w.shape[2] == ksize
        y = F.conv2d(a16.permute(0, 3, 1, 2), w, b, padding=ksize // 2).permute(0, 2, 3, 1)
        if residual is not None:
            assert residual.shape == y.shape
            y = y + residual
        return y.contiguous()

    @staticmethod
    def _attn(qkv, B, N, heads, d):
        hid = heads * d
        q, k, v = (qkv[:, i * hid:(i + 1) * hid].reshape(B, N, heads, d).permute(0, 2, 1, 3) for i in range(3))
        w = torch.softmax(q @ k.transpose(-1, -2) / math.sqrt(d), dim=-1)
        return (w @ v).permute(0, 2, 1, 3).reshape(B * N, hid)

    def attention(self, qkv16, B, N, heads, d):
        self.calls.append("attention")
        assert tuple(qkv16.shape) == (B * N, 3 * heads * d)
        return self._attn(qkv16, B, N, heads, d).contiguous()

    def linear(self, x, w, b, silu=False):
        assert x.is_contiguous() and w.is_contiguous() and x.shape[1] == w.shape[1] <= 1536 and b.shape == (w.shape[0],)
        y = F.linear(x, w, b)
        return F.silu(y) if silu else y

    def timestep_embedding(self, t, dim):
        assert t.dtype == torch.float64
        return timestep_embedding(t, dim)                                 # fp32 like the kernel's output

    def conv_backward(self, a16, dy16, w, ksize, need_dx=True):
        self.calls.append(f"conv_backward{ksize}")
        assert dy16.is_contiguous() and dy16.shape[:3] == a16.shape[:3] and dy16.shape[3] == w.shape[0]
        with torch.enable_grad():
            a = a16.detach().clone().requires_grad_(True)
            ww = w.detach().clone().requires_grad_(True)
            bb = torch.zeros(w.shape[0], dtype=w.dtype, requires_grad=True)
            y = F.conv2d(a.permute(0, 3, 1, 2), ww, bb, padding=ksize // 2).permute(0, 2, 3, 1)
            da, dw, db = torch.autograd.grad(y, (a, ww, bb), dy16)
        return (da if need_dx else None), dw, db

    def groupnorm_backward(self, x, dact, gamma, beta, film, silu, drop_p, seed, layer):
        self.calls.append("groupnorm_backward")
        assert x.is_contiguous() and dact.is_contiguous() and x.shape == dact.shape
        with torch.enable_grad():
            xs = x.detach().clone().requires_grad_(True)
            g = gamma.detach().clone().requires_grad_(True)
            b = beta.detach().clone().requires_grad_(True)
            f = film.detach().clone().requires_grad_(True) if film is not None else None
            y = self._gn(xs, g, b, f, silu, self._mask(x.shape, drop_p, seed, layer))
            outs = torch.autograd.grad(y, (xs, g, b) + ((f,) if f is not None else ()), dact)
        return outs[0], outs[1], outs[2], (outs[3] if f is not None else None)

    def attention_backward(self, qkv, do, B, N, heads, d):
        self.calls.append("attention_backward")
        with torch.enable_grad():
            q = qkv.detach().clone().requires_grad_(True)
            (dq,) = torch.autograd.grad(self._attn(q, B, N, heads, d), (q,), do)
        return dq


@pytest.fixture
def contract_ops(monkeypatch):
    """Every graph built inside the test gets this ContractOps instance instead of KernelOps (the package itself has no switch)."""
    import v_diffusion_b200.training as T
    ops = ContractOps()
    monkeypatch.setattr(T, "KernelOps", lambda operand_dtype="fp16": ops)
    return ops


def _build(cfg, seed, drop_rate=0.0):
    sd = make_state_dict(cfg, seed)
    net = UNet(cfg["in_channels"], cfg["hid_channels"], cfg["out_channels"], cfg["ch_multipliers"], cfg["num_res_blocks"],
               cfg["apply_attn"], embedding_dim=cfg["embedding_dim"], drop_rate=drop_rate, head_dim=cfg["head_dim"],
               num_heads=cfg["num_heads"], num_classes=cfg["num_classes"], multitags=cfg["multitags"])
    net.load_state_dict(sd, strict=True)
    return sd, net.double()


GRAPH_CASES = {
    # two levels: channel-changing blocks with 1x1 skips, an avg-pool and a nearest-upsample block, concat widths 192 / 256 / 128 (two channels per group at the narrowest),
    # attention on the inner level, class-conditional with an unconditional row (label 0)
    "two_level_cond": dict(cfg=_cfg(hid=64, mult=(1, 2), nrb=2, attn=(False, True), num_classes=10), res=8, B=3, labels=[0, 3, 10]),
    # three levels, attention inside the resampling blocks, explicit head_dim, 6 output channels ("both"), no labels
    "three_level_hd": dict(cfg=_cfg(hid=64, out_channels=6, mult=(1, 1, 2), nrb=1, attn=(False, True, True), embedding_dim=96,
                                    head_dim=32, num_heads=None), res=16, B=2, labels=None),
    # multi-hot labels (CelebA attributes), single-channel images
    "multitag": dict(cfg=_cfg(in_channels=1, out_channels=1, hid=64, mult=(1, 1), nrb=1, attn=(True, False), num_classes=5,
                              multitags=True), res=8, B=3, labels="multitag"),
}


@pytest.mark.parametrize("name", sorted(GRAPH_CASES))
def test_graph_orchestration_matches_autograd(name, contract_ops):
    """Output and EVERY parameter gradient of the composed forward / backward (fp64 contract model in place of the kernels)
    against torch autograd through the oracle UNet (fp32) for d (sum of out * go)."""
    case = GRAPH_CASES[name]
    cfg, B, R = case["cfg"], case["B"], case["res"]
    sd, net = _build(cfg, seed=5)
    g = torch.Generator().manual_seed(99)
    x = torch.randn(B, cfg["in_channels"], R, R, generator=g)
    t = torch.rand(B, generator=g, dtype=torch.float64)
    go = torch.randn(B, cfg["out_channels"], R, R, generator=g)
    if case["labels"] == "multitag":
        y = (torch.rand(B, cfg["num_classes"], generator=g) > 0.5).float()
        y[0] = 0                                                           # a row without any tag: clamp(min=1) path
    elif case["labels"] is not None:
        y = torch.tensor(case["labels"])
    else:
        y = None
    ops = contract_ops
    graph = UNetTrainGraph(net)
    out = graph.forward(x.double(), t, y)
    grads = graph.backward(go.double())

    ref_sd = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    with torch.enable_grad():
        ref = _unet_forward(ref_sd, cfg, x, t, y, None)
        ref.backward(go)
    assert out.shape == ref.shape

    def rel(a, b):
        return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()
    assert rel(out, ref.detach()) < 2e-5, rel(out, ref.detach())
    assert set(grads) == set(sd)
    worst = {}
    for k in sd:
        want = ref_sd[k].grad
        if want is None:                                                   # class_embed with y = None
            assert not grads[k].any(), k
            continue
        assert grads[k].shape == want.shape, k
        # (+ an absolute floor for the fp32 reference's own rounding: with one channel per group a bias in front of a
        # GroupNorm has an analytically zero gradient -- fp64 here gives ~1e-16, fp32 autograd ~1e-6)
        worst[k] = (grads[k].double() - want.double()).norm().item() / (want.double().norm().item() + 2e-5 * math.sqrt(want.numel()))
    bad = {k: v for k, v in worst.items() if v > 2e-4}
    assert not bad, bad
    # every kernel family took part
    for fam in ("groupnorm", "groupnorm_train", "conv1", "conv3", "attention", "conv_backward1", "conv_backward3",
                "groupnorm_backward", "attention_backward"):
        assert fam in ops.calls, fam


def test_graph_dropout_uses_one_stream_for_forward_and_backward(contract_ops):
    """.train() with drop_rate > 0: the backward regenerates the forward's masks from (seed, layer); the gradient is the one
    autograd gives for the same masks (checked by finite differences on one weight), and a different seed changes the output."""
    cfg = _cfg(hid=32, mult=(1, 2), nrb=1, attn=(False, True), num_classes=0)
    sd, net = _build(cfg, seed=8, drop_rate=0.3)
    net.train()
    g = torch.Generator().manual_seed(3)
    x = torch.randn(2, 3, 8, 8, generator=g).double()
    t = torch.rand(2, generator=g, dtype=torch.float64)
    go = torch.randn(2, 3, 8, 8, generator=g).double()
    graph = UNetTrainGraph(net)
    out = graph.forward(x, t, None, seed=1234)
    grads = graph.backward(go)
    again = graph.forward(x, t, None, seed=1234)
    graph.backward(go)
    assert torch.equal(out, again)
    other = graph.forward(x, t, None, seed=1235)
    graph.backward(go)
    assert (other - out).abs().max() > 1e-3
    net.eval()                                                             # eval: dropout off (drop_rate read only in .train())
    off = graph.forward(x, t, None, seed=1234)
    graph.backward(go)
    assert (off - out).abs().max() > 1e-3
    net.train()
    # finite difference on one scalar of a mid-network weight
    key, idx = "middle.0.conv1.weight", (3, 5, 1, 2)
    p = dict(net.named_parameters())[key]
    eps = 1e-6
    with torch.no_grad():
        p[idx] += eps
        up = (graph.forward(x, t, None, seed=1234) * go).sum()
        graph.backward(go)
        p[idx] -= 2 * eps
        dn = (graph.forward(x, t, None, seed=1234) * go).sum()
        graph.backward(go)
        p[idx] += eps
    fd = ((up - dn) / (2 * eps)).item()
    assert abs(fd - grads[key][idx].item()) <= 1e-5 * max(1.0, abs(fd)), (fd, grads[key][idx].item())


def test_block_list_matches_oracle_plan():
    """The block order read off the product's module tree equals the oracle's restatement of unet.py:250-283, 297-321."""
    from oracle.unet_ref import block_plan
    for cfg in (_cfg(hid=32, mult=(1, 2), nrb=2, attn=(False, True)), _cfg(hid=32, mult=(1, 1, 2), nrb=1, attn=(False, True, True)),
                _cfg(hid=32, mult=(1, 2, 2, 3), nrb=3, attn=(True, False, True, True)), _cfg(hid=32, mult=(2,), nrb=1, attn=(True,))):
        _, net = _build(cfg, seed=1)
        got = [(b["kind"], b["name"], {0: "none", 1: "down", 2: "up"}[b["resample"]], b["concat"], b["push"]) for b in block_list(net)]
        want = [(b["kind"], b["name"], b["resample"], b["concat"], b["push"]) for b in block_plan(cfg)]
        assert got == want


def test_resample_adjoints():
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 4, 6, 5, generator=g, dtype=torch.float64, requires_grad=True)
    for mode, fn in ((1, lambda z: F.avg_pool2d(z, 2)), (2, lambda z: F.interpolate(z, scale_factor=2, mode="nearest"))):
        y = fn(x.permute(0, 3, 1, 2)).permute(0, 2, 3, 1)
        go = torch.randn(y.shape, generator=g, dtype=torch.float64)
        (want,) = torch.autograd.grad(y, (x,), go)
        assert torch.allclose(_resample_adjoint(go, mode), want, atol=1e-12)
    assert _resample_adjoint(x, 0) is x


def test_pow2_scale_keeps_tiny_gradients_in_fp16_range():
    """d loss.mean() / d activations of order 1e-7 flush to zero in fp16; scaled by the power of two they keep ~11 bits."""
    g = torch.Generator().manual_seed(1)
    x = torch.randn(4096, generator=g) * 3e-8
    s = pow2_scale_for_16bit(x)
    assert math.log2(s.item()) == round(math.log2(s.item()))              # an exact power of two
    assert 1024 <= (x * s).abs().max().item() < 2048
    back = (x * s).to(torch.float16).float() / s
    plain = x.to(torch.float16).float()
    assert ((back - x).norm() / x.norm()).item() < 1e-3
    assert ((plain - x).norm() / x.norm()).item() > 0.2                   # what the scaling is for
    assert pow2_scale_for_16bit(torch.zeros(8)).item() == 1.0
    assert pow2_scale_for_16bit(torch.tensor([float("inf"), 1.0])).item() == 1.0


def _reducer_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        g = torch.Generator().manual_seed(100 + rank)
        shapes = {"a.weight": (7, 5, 3, 3), "a.bias": (7,), "b.weight": (300, 11), "c": (1,), "d.weight": (64, 64)}
        grads = {k: torch.randn(s, generator=g) for k, s in shapes.items()}
        red = GradBucketReducer(world, bucket_bytes=4096)                   # several buckets, one of them oversize
        for k, v in grads.items():
            red.add(k, v.clone())
        out = red.finish()
        # numpy copies: a torch tensor in a Queue is a shared-memory handle that dies with this process
        q.put((rank, {k: v.numpy().copy() for k, v in grads.items()}, {k: v.numpy().copy() for k, v in out.items()}))
        dist.barrier()
    finally:
        dist.destroy_process_group()


def test_grad_bucket_reducer_averages_over_ranks_gloo():
    """World size 2 over gloo: every rank ends with the mean of the two ranks' gradients, shapes and names preserved."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_reducer_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = [q.get(timeout=120) for _ in range(2)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    got.sort(key=lambda e: e[0])
    (_, g0, o0), (_, g1, o1) = got
    import numpy as np
    for k in g0:
        mean = (g0[k] + g1[k]) / 2
        assert o0[k].shape == g0[k].shape
        assert np.allclose(o0[k], mean, atol=1e-7) and np.array_equal(o0[k], o1[k]), k


def test_grad_bucket_reducer_single_rank_is_identity():
    red = GradBucketReducer(1, bucket_bytes=64)
    a, b = torch.arange(6.).reshape(2, 3), torch.ones(40)
    red.add("a", a); red.add("b", b)
    out = red.finish()
    assert torch.equal(out["a"], a) and torch.equal(out["b"], b)
    assert red.finish() == {}


def test_kernel_ops_is_the_only_product_backend():
    """No fallback, no switch: a graph always builds KernelOps (tests can only monkeypatch the name), and KernelOps refuses
    CPU tensors."""
    import inspect
    from v_diffusion_b200.training import TrainingStep
    assert list(inspect.signature(UNetTrainGraph.__init__).parameters) == ["self", "model"]
    assert "ops" not in " ".join(inspect.signature(TrainingStep.__init__).parameters)
    from v_diffusion_b200.training import KernelOps
    cfg = _cfg(hid=32, mult=(1,), nrb=1, attn=(False,))
    _, net = _build(cfg, seed=1)
    graph = UNetTrainGraph(net.float())
    assert isinstance(graph.ops, KernelOps)
    with pytest.raises((ValueError, RuntimeError)):
        graph.forward(torch.zeros(1, 3, 8, 8), torch.zeros(1, dtype=torch.float64))
    with pytest.raises(NotImplementedError):
        KernelOps("fp16x3")


def test_kernel_ops_marshals_every_call(monkeypatch):
    """Without a GPU every KernelOps method must still get through ctypes (arity and types against _lib's argtypes) and come
    back with the library's own CUDA error -- not a ctypes ArgumentError / TypeError, and never a silent success."""
    if torch.cuda.is_available():
        pytest.skip("meant for the CPU-only container")
    from v_diffusion_b200 import _lib
    from v_diffusion_b200.training import KernelOps
    monkeypatch.setattr(_lib, "current_stream_ptr", lambda: None)
    monkeypatch.setattr(KernelOps, "_cuda32", staticmethod(lambda *a: None))
    ops = KernelOps("fp16")
    B, H, W, Cc = 2, 8, 8, 128
    x, g, b, film = torch.zeros(B, H, W, Cc), torch.ones(Cc), torch.zeros(Cc), torch.zeros(B, 2 * Cc)
    a16, w3, w1 = torch.zeros(B, H, W, Cc, dtype=torch.float16), torch.zeros(Cc, Cc, 3, 3), torch.zeros(Cc, Cc, 1, 1)
    calls = {
        "groupnorm": lambda: ops.groupnorm(x, None, g, b, None, True, 0, True, False),
        "groupnorm concat": lambda: ops.groupnorm(x, x, torch.ones(2 * Cc), torch.zeros(2 * Cc), torch.zeros(B, 4 * Cc), True, 1, True, True),
        "groupnorm_train": lambda: ops.groupnorm_train(x, g, b, film, 0.2, 5, 3),
        "groupnorm_train p=0": lambda: ops.groupnorm_train(x, g, b, film, 0.0, 5, 3),
        "conv": lambda: ops.conv(a16, w3, b, x, 3),
        "conv out16": lambda: ops.conv(a16, w1, b, None, 1, out16=True),
        "attention": lambda: ops.attention(torch.zeros(B * 64, 3 * Cc, dtype=torch.float16), B, 64, 1, Cc),
        "linear": lambda: ops.linear(torch.zeros(B, 64), torch.zeros(32, 64), torch.zeros(32), True),
        "conv_backward": lambda: ops.conv_backward(a16, a16, w3, 3),
        "conv_backward wgrad only": lambda: ops.conv_backward(a16, a16, w1, 1, need_dx=False),
        "groupnorm_backward": lambda: ops.groupnorm_backward(x, x, g, b, film, True, 0.2, 5, 3),
        "attention_backward": lambda: ops.attention_backward(torch.zeros(B * 64, 3 * Cc), torch.zeros(B * 64, Cc), B, 64, 1, Cc),
    }
    for name, fn in calls.items():
        with pytest.raises(RuntimeError, match="vdt_b200: "):
            fn()
    with pytest.raises(ValueError):
        ops.timestep_embedding(torch.zeros(B, dtype=torch.float64), 64)       # CPU tensor refused before the call


def test_ctypes_argtypes_have_the_headers_arity():
    """Every prototype in include/vdt_b200.h against the argtypes _lib.py declares: same number of parameters."""
    import re
    from v_diffusion_b200 import _lib
    L = _lib.lib()
    hdr = re.sub(r"/\*.*?\*/", "", open(_lib.INCLUDE).read(), flags=re.S)
    protos = re.findall(r"\b(vdt_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", hdr, flags=re.S)
    assert len(protos) >= 40
    for name, params in protos:
        n = 0 if params.strip() in ("", "void") else params.count(",") + 1
        at = getattr(L, name).argtypes
        if at is None:
            assert n == 0, f"{name}: {n} parameters in the header, no argtypes in _lib.py"
        else:
            assert len(at) == n, f"{name}: header has {n} parameters, _lib.py declares {len(at)}"


def test_autograd_mode_runs_the_reference_training_lines_unchanged(contract_ops):
    """UNet.autograd = True: the reference's own step -- loss = diffusion.train_loss(model, x_0, t, y, noise).mean();
    loss.backward(); clip_grad_norm_; optimizer.step() (train_utils.py:137-163) -- written against this module exactly as
    against the reference's, leaves in every .grad what autograd through the oracle UNet leaves (contract stand-in for the
    kernels), and torch.optim.AdamW then moves the parameters identically."""
    cfg = _cfg(hid=64, mult=(1, 2), nrb=1, attn=(False, True), num_classes=10)
    sd, net = _build(cfg, seed=4)
    net.autograd = True
    net.train()
    g = torch.Generator().manual_seed(12)
    x0 = torch.randn(3, 3, 8, 8, generator=g).clamp(-1, 1)
    t = torch.rand(3, generator=g, dtype=torch.float64)
    noise = torch.randn(3, 3, 8, 8, generator=g)
    y = torch.tensor([2, 0, 9])
    from oracle import train_loss as oracle_train_loss

    def run(denoise_fn, params):
        opt = torch.optim.AdamW(params, lr=2e-4, weight_decay=0.001)
        per, _ = oracle_train_loss(denoise_fn, x0, t, y.clone(), noise, model_out_type="v", reweight_type="snr_trunc")
        loss = per.mean()
        loss.backward()
        total = torch.nn.utils.clip_grad_norm_(params, max_norm=1.0)
        opt.step()
        return float(loss.detach()), float(total)

    mine = run(lambda a, b, c: net(a.double(), b, c).float(), list(net.parameters()))
    ref_p = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    ref = run(lambda a, b, c: _unet_forward(ref_p, cfg, a, b, c, None), list(ref_p.values()))
    assert abs(mine[0] - ref[0]) <= 1e-5 * abs(ref[0]) and abs(mine[1] - ref[1]) <= 1e-4 * ref[1], (mine, ref)
    for k, p in net.named_parameters():
        assert p.grad is not None and p.grad.shape == p.shape, k
        step_mine, step_ref = p.detach().float() - sd[k], ref_p[k].detach() - sd[k]
        # AdamW's first step is lr * g / (|g| + eps): entries with |g| ~ 1e-8 are sensitive to the last bit of g, the rest are not
        d = (step_mine - step_ref).abs()
        assert d.mean() <= 1e-6 and (d > 2e-5).float().mean() <= 1e-3 and d.max() <= 4.1e-4, (k, d.mean().item(), d.max().item())
    # without grad mode (sampling) or with autograd off, forward() stays the plan path, which refuses a CPU tensor
    net.autograd = False
    with pytest.raises(RuntimeError, match="CUDA"):
        net(x0, t, y)


def test_reference_train_loss_drives_the_autograd_unet(contract_ops, golden_dir):
    """This package's UNet (autograd mode, contract stand-in for the kernels) as the denoise_fn of train_loss, then
    loss.mean().backward() as in Trainer.step: the per-sample loss and every parameter's gradient against what the UNMODIFIED
    reference's own UNet + GaussianDiffusion.train_loss + autograd produced on the same seeded inputs
    (tests/golden/train_grads_small.npz, made by tests/golden/make_train_grad_golden.py).  train_loss is the oracle's
    restatement, which test_oracle_golden.py pins to the reference's on its own fixtures."""
    import numpy as np
    from oracle import train_loss
    from tests.cases import TRAIN_GRAD_CASE, build_train_grad_inputs, grad_probe
    case = TRAIN_GRAD_CASE
    g = np.load(os.path.join(golden_dir, "train_grads_small.npz"))
    _, net = _build(case["cfg"], case["wseed"])
    net.autograd = True
    net.train()
    x0, t, noise, y = build_train_grad_inputs(case)
    loss, _ = train_loss(lambda a, b, c: net(a.double(), b, c).float(), x0, t, y.clone(), noise,
                         model_out_type=case["model_out_type"], reweight_type=case["reweight_type"])
    assert loss.shape == (case["B"],)
    loss.mean().backward()
    np.testing.assert_allclose(loss.detach().numpy(), g["loss"], rtol=1e-5)
    params = dict(net.named_parameters())
    names = [str(n) for n in g["names"]]
    assert sorted(names) == sorted(params)
    for k in names:
        gr = params[k].grad.double()
        n_ref = float(g["norm/" + k])
        assert abs(gr.norm().item() - n_ref) <= 1e-4 * n_ref + 1e-9, k
        assert abs((gr * grad_probe(k, gr.shape)).sum().item() - float(g["proj/" + k])) <= 1e-3 * n_ref + 1e-9, k
        if ("full/" + k) in g.files:
            assert (gr - torch.from_numpy(g["full/" + k]).double()).norm().item() <= 1e-4 * n_ref + 1e-9, k


def test_gpu_worker_and_bench_block_dry_run():
    """tests/train_step_worker.py (the GPU suite's child process) and bench.py's train_step block, run here on the CPU with
    stand-ins for everything that needs a device (scripts/dryrun_train_worker.py): guards their host logic against bit-rot."""
    import subprocess
    r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "dryrun_train_worker.py")], cwd=ROOT, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0 and "dry run OK" in r.stdout, r.stdout[-1500:] + r.stderr[-1500:]


def test_two_rank_training_step_dry_run_gloo():
    """tests/train_step_ddp_worker.py (the two-GPU NCCL case of the GPU suite) on the CPU: two processes over gloo with the
    same stand-ins -- loss reduce, bucketed gradient average, optimizer on every rank, EMA on the leader only; the replicas'
    parameters stay bit-identical over three steps on different data, and they move."""
    import json
    import subprocess
    port = 29800 + (os.getpid() % 1000)
    procs = []
    for rank in range(2):
        env = dict(os.environ, RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, "scripts", "dryrun_train_worker.py"), "ddp"], cwd=ROOT, env=env,
                                      stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    outs = [p.communicate(timeout=600) for p in procs]
    assert all(p.returncode == 0 for p in procs), "\\n".join(o[1][-1500:] for o in outs)
    lines = [ln for ln in outs[0][0].splitlines() if ln.startswith("RESULT ")]
    assert lines, outs[0][0][-1000:]
    res = json.loads(lines[-1][len("RESULT "):])
    assert res["identical"] and res["finite"] and 0 < res["moved"] < 1e-2, res


def test_ema_weights_context_swaps_and_restores():
    """``with step.ema():`` (the reference's ``with self.ema:``, utils.py:151-166): shadow in, live weights back out -- also
    when the block raises -- and the model's plan cache is invalidated on both edges."""
    from v_diffusion_b200.training import ema_weights
    cfg = _cfg(hid=32, mult=(1,), nrb=1, attn=(False,))
    _, net = _build(cfg, seed=2)
    live = {k: p.detach().clone() for k, p in net.named_parameters()}
    shadow = {k: v + 1.0 for k, v in live.items()}
    e0 = net._weights_epoch
    with ema_weights(net, shadow) as m:
        assert m is net and net._weights_epoch == e0 + 1
        assert all(torch.equal(p, shadow[k]) for k, p in net.named_parameters())
    assert net._weights_epoch == e0 + 2
    assert all(torch.equal(p, live[k]) for k, p in net.named_parameters())
    with pytest.raises(ZeroDivisionError):
        with ema_weights(net, shadow):
            1 / 0
    assert all(torch.equal(p, live[k]) for k, p in net.named_parameters())
    with pytest.raises(RuntimeError, match="no EMA shadow"):
        with ema_weights(net, {}):
            pass


def test_adamw_state_round_trips_through_torch_format():
    """Checkpoint interop (train_utils.py:309-352): the moments leave and enter in torch.optim.AdamW.state_dict() form --
    a state read from a real torch AdamW and written back loads into a fresh torch AdamW that then steps identically."""
    from v_diffusion_b200.optim import torch_adamw_state, read_torch_adamw_state, strip_module_prefix
    g = torch.Generator().manual_seed(4)
    shapes = {"a.weight": (5, 3, 3, 3), "a.bias": (5,), "b.weight": (7, 4)}
    names = list(shapes)

    def fresh():
        gg = torch.Generator().manual_seed(9)
        ps = [torch.nn.Parameter(torch.randn(s, generator=gg)) for s in shapes.values()]
        return ps, torch.optim.AdamW(ps, lr=2e-4, betas=(0.9, 0.999), weight_decay=0.001)

    def run(ps, opt, n, seed):
        gg = torch.Generator().manual_seed(seed)
        for _ in range(n):
            for p in ps:
                p.grad = torch.randn(p.shape, generator=gg)
            opt.step()
    p1, o1 = fresh()
    assert read_torch_adamw_state(o1.state_dict(), names)[2] == 0                  # fresh optimizer: no state yet
    run(p1, o1, 3, 1)
    exp_avg, exp_avg_sq, step, group = read_torch_adamw_state(o1.state_dict(), names)
    assert step == 3 and group["lr"] == 2e-4 and set(exp_avg) == set(names)
    emitted = torch_adamw_state(names, exp_avg, exp_avg_sq, step, group["lr"], group["betas"], group["eps"], group["weight_decay"])
    p2, o2 = fresh()
    with torch.no_grad():
        for a, b in zip(p2, p1):
            a.copy_(b)
    import copy
    o2.load_state_dict(copy.deepcopy(emitted))            # (torch's load_state_dict keeps same-dtype tensors by reference)
    run(p1, o1, 2, 2)
    run(p2, o2, 2, 2)
    assert all(torch.equal(a, b) for a, b in zip(p1, p2))
    assert strip_module_prefix({"module.x.weight": 1, "y": 2}) == {"x.weight": 1, "y": 2}
    bad = o1.state_dict()
    bad["param_groups"].append(dict(bad["param_groups"][0]))
    with pytest.raises(RuntimeError, match="single AdamW parameter group"):
        read_torch_adamw_state(bad, names)


def test_bench_train_step_block_never_breaks_the_bench_line():
    """bench.py's train_step block runs in a child process; when the child fails (here: no GPU) the block comes back as an
    {"error": ...} entry instead of an exception, so the headline JSON line is still printed."""
    if torch.cuda.is_available():
        pytest.skip("meant for the CPU-only container")
    import bench
    out = bench.train_step_block(timeout_s=120)
    assert set(out) == {"error"} and "child rc=" in out["error"], out


def test_bench_dump_outputs_is_float32_and_a_fixed_sample_under_the_cap(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float32 whatever the input dtype; above the size cap, the same seeded subset of the images on
    every call, kept in batch order."""
    import numpy as np
    import bench
    x = torch.randn(12, 3, 8, 8, generator=torch.Generator().manual_seed(3), dtype=torch.float64)
    bench.dump_outputs(str(tmp_path / "all"), x)
    full = np.load(tmp_path / "all" / "samples.npy")
    assert full.dtype == np.float32 and np.array_equal(full, x.float().numpy())
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 5 * x[0].numel() * 4)
    bench.dump_outputs(str(tmp_path / "a"), x)
    bench.dump_outputs(str(tmp_path / "b"), x)
    a, b = np.load(tmp_path / "a" / "samples.npy"), np.load(tmp_path / "b" / "samples.npy")
    assert a.shape == (5, 3, 8, 8) and np.array_equal(a, b)
    rows = [next(i for i in range(12) if np.array_equal(full[i], r)) for r in a]
    assert rows == sorted(rows) and len(set(rows)) == 5
