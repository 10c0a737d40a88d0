"""GPU parity of wgrad on feature maps whose forward-conv tile holds fewer than 128 pixels (28², 14², 7², 24², 12², 6², 5²),
through the C ABI, with the method and bars of test_conv_backward_vs_autograd (tests/test_gpu_kernels.py).

In wgrad the pixels are the contraction, so shared-memory rows past a tile's last pixel must be zero in both operands.  Each case
first runs one full-tile wgrad on large finite inputs, which leaves large values in the shared memory of the SMs it ran on; a
ragged call that read stale rows would then miss the bars.  This is a best-effort guard, not a proof: nothing makes a later CTA
land on an SM whose shared memory still holds those values.
"""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DT = {1: torch.float16, 0: torch.bfloat16}


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


def _dirty_shared_memory(L, f16):
    """One full-tile wgrad (32², 128 pixels per tile, 256 -> 256, every operand chunk of both stages loaded) on ~1e4-scale
    inputs."""
    g = torch.Generator(device="cuda").manual_seed(1)
    x = (torch.randn(2, 32, 32, 256, device="cuda", generator=g) * 1e4).to(DT[f16])
    dy = (torch.randn(2, 32, 32, 256, device="cuda", generator=g) * 1e4).to(DT[f16])
    dw = torch.empty(256, 256, 3, 3, device="cuda")
    _check(L, L.vdt_op_conv_wgrad(_p(x), _p(dy), 2, 32, 32, 256, 256, 3, _p(dw), None, f16, None))
    torch.cuda.synchronize()


RAGGED_CASES = [
    # B, H, cin, cout, k      pixels per tile
    (2, 28, 256, 256, 3),     # 112: 4 rows of 28, 7 MMAs per tap, none wasted (configs[3] level 0)
    (3, 28, 256, 128, 1),     # 112, 1x1
    (4, 14, 256, 256, 3),     # 98: 7 rows of 14 (configs[3] level 1)
    (3, 7, 256, 256, 3),      # 98: two images per tile, odd batch -> the last tile's second image is out of bounds (level 2)
    (7, 5, 128, 128, 3),      # 125: five images per tile, the last tile holds two
    (5, 6, 128, 128, 3),      # 108: three images per tile, ragged batch
    (3, 12, 128, 256, 3),     # 72: 6 rows of 12, 5 MMAs per tap
    (2, 24, 192, 128, 3),     # 96: 4 rows of 24, 192-wide input-channel block
    (2, 28, 192, 192, 3),     # 112 together with the 64-channel tail block of cout 192
    (2, 28, 512, 256, 3),     # 112, two input-channel blocks (configs[3] concat conv1)
]


@pytest.mark.parametrize("f16", [1, 0])
@pytest.mark.parametrize("B,H,cin,cout,k", RAGGED_CASES)
def test_ragged_wgrad_vs_autograd(L, B, H, cin, cout, k, f16):
    """wgrad (+ bias grad) on a ragged tile against torch autograd in fp64 on the same 16-bit operands: dW within 1e-4, db
    within 1e-5 rel-L2, every dW entry written, a second call bit-identical."""
    g = torch.Generator(device="cuda").manual_seed(H + cin + cout + k)
    x = torch.randn(B, H, H, cin, device="cuda", generator=g).to(DT[f16])
    dy = torch.randn(B, H, H, cout, device="cuda", generator=g).to(DT[f16])
    _dirty_shared_memory(L, f16)
    dw = torch.full((cout, cin, k, k), float("nan"), device="cuda")      # every entry must be written
    db = torch.zeros(cout, device="cuda")
    _check(L, L.vdt_op_conv_wgrad(_p(x), _p(dy), B, H, H, cin, cout, k, _p(dw), _p(db), f16, None))
    torch.cuda.synchronize()
    xd = x.double().permute(0, 3, 1, 2)
    wd = torch.zeros(cout, cin, k, k, device="cuda", dtype=torch.float64, requires_grad=True)
    bd = torch.zeros(cout, device="cuda", dtype=torch.float64, requires_grad=True)
    F.conv2d(xd, wd, bd, padding=k // 2).backward(dy.double().permute(0, 3, 1, 2))
    print(f"wgrad {cin}->{cout} k{k} @{H}x{H} B={B}: wgrad rel {_rel(dw, wd.grad):.2e} dbias rel {_rel(db, bd.grad):.2e}")
    assert bool(torch.isfinite(dw).all())
    assert _rel(dw, wd.grad) <= 1e-4
    assert _rel(db, bd.grad) <= 1e-5
    dw2 = torch.zeros_like(dw)
    _check(L, L.vdt_op_conv_wgrad(_p(x), _p(dy), B, H, H, cin, cout, k, _p(dw2), None, f16, None))
    torch.cuda.synchronize()
    assert torch.equal(dw, dw2)


@pytest.mark.parametrize("f16", [1, 0])
@pytest.mark.parametrize("hid", [256, 64])
def test_in_conv_patch_gemm_wgrad_at_28(L, hid, f16):
    """in_conv's weight gradient as the training step computes it (training.py): a 1x1 GEMM over the 3x3 patches of a
    1-channel 28x28 image, K = 9 real columns padded to 128; hid 256 is configs[3]'s network, hid 64 the small MNIST-style one."""
    B, R, K = 3, 28, 128
    g = torch.Generator(device="cuda").manual_seed(hid + f16)
    img = torch.randn(B, 1, R, R, device="cuda", generator=g)
    cols = F.pad(F.unfold(img, 3, padding=1).transpose(1, 2), (0, K - 9)).reshape(B, R, R, K).contiguous().to(DT[f16])
    dy = torch.randn(B, R, R, hid, device="cuda", generator=g).to(DT[f16])
    _dirty_shared_memory(L, f16)
    dw = torch.full((hid, K, 1, 1), float("nan"), device="cuda")
    db = torch.zeros(hid, device="cuda")
    _check(L, L.vdt_op_conv_wgrad(_p(cols), _p(dy), B, R, R, K, hid, 1, _p(dw), _p(db), f16, None))
    torch.cuda.synchronize()
    ref = torch.einsum("bhwc,bhwk->ck", dy.double(), cols.double()).reshape(hid, K, 1, 1)
    ref_db = dy.double().sum(dim=(0, 1, 2))
    print(f"in_conv wgrad hid {hid} @28 f16={f16}: wgrad rel {_rel(dw, ref):.2e} (padding columns max |dW| "
          f"{dw[:, 9:].abs().max().item():.1e}) dbias rel {_rel(db, ref_db):.2e}")
    assert _rel(dw, ref) <= 1e-4
    assert not dw[:, 9:].any()                                              # zero input columns: exactly zero gradient
    assert _rel(db, ref_db) <= 1e-5
    dw2 = torch.zeros_like(dw)
    _check(L, L.vdt_op_conv_wgrad(_p(cols), _p(dy), B, R, R, K, hid, 1, _p(dw2), None, f16, None))
    torch.cuda.synchronize()
    assert torch.equal(dw, dw2)
