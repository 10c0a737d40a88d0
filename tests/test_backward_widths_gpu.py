"""GPU parity of the backward kernels at the channel widths of the CelebA and hid-64 networks, through the C ABI, with the method
and bars of test_groupnorm_backward_vs_autograd / test_conv_backward_vs_autograd (tests/test_gpu_kernels.py):

* GroupNorm backward at C % 64 == 0 beyond 128 / 256 / 512 / 1024: 2-wide channel vectors for groups of 2 / 6 / 18 / 42 channels,
  several channel blocks per sample for C > 1024 or rows that would idle a CTA; dropout regenerated from the forward's mask.
* wgrad with cout % 128 == 64: the last output-channel block holds 64 channels.
"""
import ctypes as C
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DT = {1: torch.float16, 0: torch.bfloat16}
EPS = {1: 0.25, 0: 1.0}              # rounding unit of the 16-bit operand formats relative to bf16


@pytest.fixture(scope="module")
def L():
    from v_diffusion_b200 import _lib
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return _lib.lib()


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _check(L, rc):
    assert rc == 0, L.vdt_last_error().decode()


def _rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-300)).item()


GN_BWD_CASES = [
    # B, H, W, C, film, silu, drop_p
    (3, 16, 16, 64, True, 1, 0.0),       # hid 64: 2-channel groups
    (2, 16, 16, 64, False, 0, 0.0),
    (2, 32, 32, 192, True, 1, 0.0),      # CelebA level 0 (6-channel groups); hid-64 concat width
    (3, 16, 16, 192, False, 0, 0.0),
    (3, 16, 16, 192, True, 1, 0.1),      # CelebA level-0 norm2 in training mode: 2-wide dropout words
    (2, 16, 16, 576, True, 1, 0.0),      # CelebA level 2: 18-channel groups, four channel blocks
    (2, 7, 9, 576, False, 0, 0.0),       # odd pixel count per slab
    (2, 8, 8, 1344, True, 1, 0.0),       # CelebA concat width: 42-channel groups, eight channel blocks
    (2, 8, 8, 1344, False, 0, 0.0),
    (2, 8, 8, 1536, True, 1, 0.0),       # widest CelebA concat: two channel blocks of 192 four-wide vectors
    (3, 8, 8, 1536, False, 0, 0.0),
]


@pytest.mark.parametrize("case", GN_BWD_CASES)
def test_groupnorm_backward_widths_vs_autograd(L, case):
    """Backward of GroupNorm(32, 1e-6) -> FiLM -> SiLU -> dropout against fp64 autograd through F.group_norm / F.silu with the
    forward kernel's own dropout mask (vdt_op_groupnorm_dropout): grad_x, grad_gamma, grad_beta and the FiLM gradients within
    2e-5; two runs bit-identical."""
    B, H, W, Cc, film_on, silu, p = case
    g = torch.Generator(device="cuda").manual_seed(19 + Cc)
    x = torch.randn(B, H, W, Cc, device="cuda", generator=g) * 1.3 + 0.4
    gamma = torch.rand(Cc, device="cuda", generator=g) + 0.5
    beta = torch.randn(Cc, device="cuda", generator=g) * 0.2
    film = (torch.randn(B, 2 * Cc, device="cuda", generator=g) * 0.3) if film_on else None
    go = torch.randn(B, H, W, Cc, device="cuda", generator=g)
    seed, layer = 7654321, 5
    mask = None
    if p > 0:
        out = torch.zeros(B, H, W, Cc, device="cuda", dtype=torch.float16)
        _check(L, L.vdt_op_groupnorm_dropout(_p(x), Cc, B, H, W, _p(gamma), _p(beta), 0, _p(out), 1, C.c_float(p), seed, layer, None))
        torch.cuda.synchronize()
        mask = (out != 0).double() / (1 - p)
        frac = 1.0 - (out != 0).float().mean().item()
        assert abs(frac - p) < 0.02, frac
    xd = x.double().requires_grad_(True)
    gd, bd = gamma.double().requires_grad_(True), beta.double().requires_grad_(True)
    fd = film.double().requires_grad_(True) if film_on else None
    y = F.group_norm(xd.permute(0, 3, 1, 2), 32, gd, bd, 1e-6).permute(0, 2, 3, 1)
    if film_on:
        y = y * (1 + fd[:, Cc:].view(B, 1, 1, Cc)) + fd[:, :Cc].view(B, 1, 1, Cc)
    if silu:
        y = F.silu(y)
    if mask is not None:
        y = y * mask
    (y * go.double()).sum().backward()

    def run():
        gx = torch.empty_like(x)
        gg, gb = torch.empty(Cc, device="cuda"), torch.empty(Cc, device="cuda")
        gf = torch.empty(B, 2 * Cc, device="cuda") if film_on else None
        _check(L, L.vdt_op_groupnorm_backward(_p(x), _p(go), Cc, B, H, W, _p(gamma), _p(beta), _p(film), silu, C.c_float(p), seed,
                                              layer, _p(gx), _p(gg), _p(gb), _p(gf), None))
        torch.cuda.synchronize()
        return [t for t in (gx, gg, gb, gf) if t is not None]

    got = run()
    want = [xd.grad, gd.grad, bd.grad] + ([fd.grad] if film_on else [])
    errs = {k: _rel(a, b) for k, a, b in zip(("x", "gamma", "beta", "film"), got, want)}
    print(f"groupnorm backward {case}: " + ", ".join(f"d{k} {v:.2e}" for k, v in errs.items()))
    assert max(errs.values()) < 2e-5, errs
    assert all(torch.equal(a, b) for a, b in zip(got, run()))    # fixed-order reductions: bit-reproducible


WGRAD_TAIL_CASES = [
    # B, H, cin, cout, k
    (2, 64, 192, 192, 3),       # CelebA level 0: one full and one 64-channel output block, 2 image rows per tile
    (2, 16, 576, 576, 3),       # CelebA level 2: four full blocks + tail, three input-channel blocks of 192
    (2, 16, 1344, 576, 3),      # CelebA concat conv1
    (2, 32, 384, 192, 1),       # 1x1 skip to 192
    (2, 16, 64, 576, 1),        # narrow input, 576 outputs
    (3, 8, 576, 576, 3),        # 8x8: two images share a tile, odd batch -> zero-filled tail tile
]


@pytest.mark.parametrize("f16", [1, 0])
@pytest.mark.parametrize("B,H,cin,cout,k", WGRAD_TAIL_CASES)
def test_conv_backward_tail_block_vs_autograd(L, B, H, cin, cout, k, f16):
    """dgrad and wgrad (+ bias grad) at cout % 128 == 64 against torch autograd in fp64 on the same 16-bit-rounded operands;
    repeated wgrad bit-identical."""
    g = torch.Generator(device="cuda").manual_seed(H + cin + cout + k)
    x = torch.randn(B, H, H, cin, device="cuda", generator=g).to(DT[f16])
    dy = torch.randn(B, H, H, cout, device="cuda", generator=g).to(DT[f16])
    w = (torch.randn(cout, cin, k, k, device="cuda", generator=g) / math.sqrt(cin * k * k))
    dx = torch.zeros(B, H, H, cin, device="cuda")
    dw = torch.full((cout, cin, k, k), float("nan"), device="cuda")      # every entry must be written
    db = torch.zeros(cout, device="cuda")
    _check(L, L.vdt_op_conv_dgrad(_p(dy), B, H, H, cin, _p(w), cout, k, _p(dx), f16, None))
    _check(L, L.vdt_op_conv_wgrad(_p(x), _p(dy), B, H, H, cin, cout, k, _p(dw), _p(db), f16, None))
    torch.cuda.synchronize()
    xd = x.double().permute(0, 3, 1, 2).requires_grad_(True)
    wd = w.to(DT[f16]).double().requires_grad_(True)
    bd = torch.zeros(cout, device="cuda", dtype=torch.float64, requires_grad=True)
    y = F.conv2d(xd, wd, bd, padding=k // 2)
    y.backward(dy.double().permute(0, 3, 1, 2))
    ref_dx = xd.grad.permute(0, 2, 3, 1)
    tail = slice(cout - 64, cout)
    print(f"conv backward {cin}->{cout} k{k} @{H}: dgrad rel {_rel(dx, ref_dx):.2e} wgrad rel {_rel(dw, wd.grad):.2e} "
          f"(tail block {_rel(dw[tail], wd.grad[tail]):.2e}) dbias rel {_rel(db, bd.grad):.2e}")
    assert _rel(dx, ref_dx) <= 2e-3 * EPS[f16] + 1e-5
    assert _rel(dw, wd.grad) <= 1e-4
    assert _rel(dw[tail], wd.grad[tail]) <= 1e-4
    assert _rel(db, bd.grad) <= 1e-5
    dw2 = torch.zeros_like(dw)
    _check(L, L.vdt_op_conv_wgrad(_p(x), _p(dy), B, H, H, cin, cout, k, _p(dw2), None, f16, None))
    torch.cuda.synchronize()
    assert torch.equal(dw, dw2)
