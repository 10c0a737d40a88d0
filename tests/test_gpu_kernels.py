"""GPU parity of each hand-written kernel, called through the C ABI (vdt_op_*), against a plain PyTorch
fp32 reference of the same op on the same (bf16-rounded) operands."""
import ctypes as C
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def L():
    from v_diffusion_b200 import _lib
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return _lib.lib()


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _check(L, rc):
    assert rc == 0, L.vdt_last_error().decode()


DT = {1: torch.float16, 0: torch.bfloat16}
# rounding unit of the 16-bit operand formats relative to bf16
EPS = {1: 0.25, 0: 1.0}


def _rel(a, b):
    return ((a.float() - b.float()).norm() / b.float().norm().clamp_min(1e-12)).item()


CONV_CASES = [
    # B, H, cin, cout, k, residual
    (2, 32, 256, 256, 3, True),
    (3, 16, 256, 256, 3, False),
    (3, 8, 256, 256, 3, True),       # two images per tile, odd batch -> zero-filled tail
    (1, 8, 128, 64, 3, False),       # single image: half-empty tile
    (2, 32, 512, 256, 3, False),
    (2, 16, 192, 64, 3, True),
    (2, 32, 64, 128, 3, False),
    (2, 32, 512, 256, 1, False),
    (3, 8, 256, 768, 1, False),      # three N tiles
    (2, 16, 128, 384, 1, False),     # N tile of 192
    (2, 64, 192, 192, 3, True),      # CelebA-style 64x64, 2 image rows per tile
    (3, 28, 64, 64, 3, True),        # MNIST 28x28: 4 image rows = 112 of the tile's 128 rows
    (3, 14, 128, 64, 3, False),      # 14x14: 7 image rows = 98 rows per tile
    (3, 7, 64, 128, 3, True),        # 7x7: two whole images = 98 rows per tile, odd image count
    (3, 14, 64, 192, 1, False),      # pointwise over 588 rows (ragged last tile)
    (5, 4, 64, 64, 3, False),        # 4x4: eight images per tile
]


@pytest.mark.parametrize("f16", [1, 0])
@pytest.mark.parametrize("B,H,cin,cout,k,res", CONV_CASES)
def test_conv_gemm(L, B, H, cin, cout, k, res, f16):
    g = torch.Generator(device="cuda").manual_seed(B * 1000 + H + cin + cout + k)
    x = torch.randn(B, cin, H, H, device="cuda", generator=g)
    w = torch.randn(cout, cin, k, k, device="cuda", generator=g) / math.sqrt(cin * k * k)
    bias = torch.randn(cout, device="cuda", generator=g)
    resid = torch.randn(B, H, H, cout, device="cuda", generator=g) if res else None
    xb = x.to(DT[f16])
    x_nhwc = xb.permute(0, 2, 3, 1).contiguous()
    out = torch.full((B, H, H, cout), float("nan"), device="cuda")
    _check(L, L.vdt_op_conv(_p(x_nhwc), B, H, H, cin, _p(w), cout, k, _p(bias), _p(resid), _p(out), f16, None, None, 4, None))
    torch.cuda.synchronize()
    ref = F.conv2d(xb.double(), w.to(DT[f16]).double(), bias.double(), padding=k // 2).permute(0, 2, 3, 1)
    if res:
        ref = ref + resid.double()
    assert torch.isfinite(out).all()
    err = (out.double() - ref).abs().max().item()
    assert err <= 2e-3, f"max abs err {err}"       # fp32 accumulation over K <= 4608 products of O(1/sqrt(K)) terms


GN_CASES = [
    # B, H, c1, c2, film, silu, resample, want_raw, want_res
    (3, 32, 256, 0, False, True, 0, False, False),
    (2, 16, 256, 256, False, True, 0, True, False),
    (2, 16, 128, 64, True, True, 0, True, False),     # 6 channels per group straddling the concat seam
    (3, 8, 256, 0, True, True, 0, False, False),
    (2, 32, 256, 0, False, True, 1, False, True),     # avg-pool
    (2, 8, 64, 0, False, True, 2, False, True),       # nearest upsample
    (2, 16, 128, 0, False, False, 0, False, False),   # attention norm: no activation
    (2, 16, 576, 0, False, True, 0, False, False),    # 18 channels per group
    (3, 28, 64, 0, True, True, 1, False, True),       # MNIST 28x28 -> 14x14 avg-pool
    (3, 14, 64, 64, False, True, 0, True, False),     # 14x14 concat
    (3, 7, 128, 0, False, True, 2, False, True),      # 7x7 -> 14x14 nearest upsample
]


@pytest.mark.parametrize("f16", [1, 0])
@pytest.mark.parametrize("B,H,c1,c2,film,silu,resample,want_raw,want_res", GN_CASES)
def test_groupnorm(L, B, H, c1, c2, film, silu, resample, want_raw, want_res, f16):
    g = torch.Generator(device="cuda").manual_seed(H * 7 + c1 + c2)
    C_ = c1 + c2
    s1 = torch.randn(B, H, H, c1, device="cuda", generator=g) * 2 + 0.5
    s2 = torch.randn(B, H, H, c2, device="cuda", generator=g) if c2 else None
    gamma = 1 + 0.2 * torch.randn(C_, device="cuda", generator=g)
    beta = 0.2 * torch.randn(C_, device="cuda", generator=g)
    stride, off = 3 * 2 * C_, 2 * C_
    ftab = torch.randn(B, stride, device="cuda", generator=g) * 0.3 if film else None
    Ho = H // 2 if resample == 1 else H * 2 if resample == 2 else H
    out_act = torch.zeros(B, Ho, Ho, C_, device="cuda", dtype=DT[f16])
    out_raw = torch.zeros(B, H, H, C_, device="cuda", dtype=DT[f16]) if want_raw else None
    out_res = torch.zeros(B, Ho, Ho, C_, device="cuda") if want_res else None
    _check(L, L.vdt_op_groupnorm(_p(s1), c1, _p(s2), c2, B, H, H, _p(gamma), _p(beta), _p(ftab), stride, off,
                                 int(silu), resample, _p(out_act), _p(out_raw), _p(out_res), f16, None, None, 4, 0, None))
    torch.cuda.synchronize()
    x = torch.cat([s1, s2], dim=3) if c2 else s1
    xn = x.permute(0, 3, 1, 2).double()
    y = F.group_norm(xn, 32, gamma.double(), beta.double(), 1e-6)
    if film:
        shift = ftab[:, off:off + C_].double()[:, :, None, None]
        scale = ftab[:, off + C_:off + 2 * C_].double()[:, :, None, None]
        y = (1 + scale) * y + shift
    if silu:
        y = F.silu(y)
    rs = (lambda z: F.avg_pool2d(z, 2)) if resample == 1 else (lambda z: F.interpolate(z, scale_factor=2, mode="nearest")) if resample == 2 else (lambda z: z)
    y = rs(y).permute(0, 2, 3, 1)
    err = (out_act.double() - y).abs().max().item()
    assert err <= 4e-2 * EPS[f16] * max(1.0, y.abs().max().item() / 4), f"act err {err}"      # 16-bit output rounding
    assert _rel(out_act, y) <= 4e-3 * EPS[f16]
    if want_raw:
        assert torch.equal(out_raw, x.to(DT[f16]))
    if want_res:
        r = rs(xn).permute(0, 2, 3, 1)
        assert (out_res.double() - r).abs().max().item() <= 1e-5


FUSED_GN_CASES = [
    # B, H, c1, c2 (second conv output concatenated), in16, film, resample
    (2, 32, 256, 0, False, True, 0),
    (3, 8, 256, 0, False, False, 0),      # 64 pixels per image: two statistics slabs
    (2, 16, 256, 256, False, False, 0),   # concat: 16 channels per group, one stats buffer per source
    (2, 32, 256, 0, True, True, 0),       # conv1 output kept in 16 bits
    (2, 16, 128, 0, False, False, 1),     # avg-pool
    (2, 8, 256, 0, False, False, 2),      # upsample
    (2, 64, 128, 0, True, False, 0),      # 4096 pixels: image split over 8 CTAs
    (2, 16, 192, 0, False, True, 0),      # 6 channels per group -> 2-column statistics entries, VEC = 2
    (2, 16, 192, 0, True, False, 0),      # same with a 16-bit input
    (2, 16, 128, 64, False, False, 0),    # concat 128 + 64: 6-channel groups straddling the seam
    (2, 8, 64, 0, False, False, 0),       # 2 channels per group
    (3, 28, 64, 0, False, True, 0),       # MNIST 28x28: tiles of 112 rows, the fourth slab of every tile half empty
    (3, 14, 128, 64, False, False, 0),    # 14x14: tiles of 98 rows (slab 3 holds 2 rows), concat seam inside a group
    (2, 28, 128, 0, True, False, 1),      # 28x28 -> 14x14 avg-pool from a 16-bit input
]


@pytest.mark.parametrize("f16", [1, 0])
@pytest.mark.parametrize("B,H,c1,c2,in16,film,resample", FUSED_GN_CASES)
def test_conv_stats_then_single_pass_groupnorm(L, B, H, c1, c2, in16, film, resample, f16):
    """conv epilogue writes partial (sum, sumsq) per 32-row slab / 4 channels; GroupNorm combines them and
    makes one pass.  Checked against torch GroupNorm of the conv output."""
    g = torch.Generator(device="cuda").manual_seed(H + c1 + c2 + in16)
    cin = 64
    sc = 4 if ((c1 + c2) // 32) % 4 == 0 else 2          # columns per statistics entry

    def conv(cout):
        x = torch.randn(B, H, H, cin, device="cuda", generator=g).to(DT[f16])
        w = torch.randn(cout, cin, 3, 3, device="cuda", generator=g) / math.sqrt(cin * 9)
        bias = torch.randn(cout, device="cuda", generator=g)
        out = torch.zeros(B, H, H, cout, device="cuda")
        out16 = torch.zeros(B, H, H, cout, device="cuda", dtype=DT[f16]) if in16 else None
        slabs = L.vdt_stat_slabs_per_image(H, H)             # 32-row quarters of the conv kernel's image-aligned M tiles
        assert slabs > 0
        stats = torch.full((B * slabs + 4, cout // sc, 2), float("nan"), device="cuda")   # + one tile of slack
        _check(L, L.vdt_op_conv(_p(x), B, H, H, cin, _p(w), cout, 3, _p(bias), None, _p(out), f16, _p(out16), _p(stats), sc, None))
        torch.cuda.synchronize()
        ref = F.conv2d(x.permute(0, 3, 1, 2).double(), w.to(DT[f16]).double(), bias.double(), padding=1).permute(0, 2, 3, 1)
        val = out16 if in16 else out
        # the statistics describe the fp32 values before any 16-bit rounding
        stats = stats[:B * slabs]
        assert torch.isfinite(stats).all()
        if (H * H) % 128 == 0 or 2 * H * H <= 128:           # full tiles: slab = 32 consecutive pixels
            rs = ref.reshape(B * H * H // 32, 32, cout // sc, sc)
            assert (stats[..., 0].double() - rs.sum(dim=(1, 3))).abs().max().item() <= 2e-3
            assert (stats[..., 1].double() - (rs * rs).sum(dim=(1, 3))).abs().max().item() <= 2e-2
        ri = ref.reshape(B, H * H, cout // sc, sc)           # any geometry: an image's slabs add up to its totals
        tot = stats.reshape(B, slabs, cout // sc, 2).double().sum(dim=1)
        assert (tot[..., 0] - ri.sum(dim=(1, 3))).abs().max().item() <= 2e-2
        assert (tot[..., 1] - (ri * ri).sum(dim=(1, 3))).abs().max().item() <= 2e-1
        return val, stats, ref

    v1, st1, r1 = conv(c1)
    v2, st2, r2 = conv(c2) if c2 else (None, None, None)
    C_ = c1 + c2
    gamma = 1 + 0.2 * torch.randn(C_, device="cuda", generator=g)
    beta = 0.2 * torch.randn(C_, device="cuda", generator=g)
    ftab = torch.randn(B, 2 * C_, device="cuda", generator=g) * 0.3 if film else None
    Ho = H // 2 if resample == 1 else H * 2 if resample == 2 else H
    out_act = torch.zeros(B, Ho, Ho, C_, device="cuda", dtype=DT[f16])
    _check(L, L.vdt_op_groupnorm(_p(v1), c1, _p(v2), c2, B, H, H, _p(gamma), _p(beta), _p(ftab), 2 * C_, 0, 1, resample,
                                 _p(out_act), None, None, f16, _p(st1), _p(st2), sc, int(in16), None))
    torch.cuda.synchronize()
    x = torch.cat([r1, r2], dim=3) if c2 else r1
    if in16:
        x = v1.double()                      # the kernel normalises the rounded values with the fp32 statistics
    y = F.group_norm(x.permute(0, 3, 1, 2), 32, gamma.double(), beta.double(), 1e-6)
    if film:
        y = (1 + ftab[:, C_:].double()[:, :, None, None]) * y + ftab[:, :C_].double()[:, :, None, None]
    y = F.silu(y)
    y = (F.avg_pool2d(y, 2) if resample == 1 else F.interpolate(y, scale_factor=2, mode="nearest") if resample == 2 else y)
    y = y.permute(0, 2, 3, 1)
    assert _rel(out_act, y) <= 4e-3 * EPS[f16] + (2e-3 if in16 else 0)


def test_statistics_layout_exists_only_for_image_aligned_slabs(L):
    assert L.vdt_stat_slabs_per_image(32, 32) == 32 and L.vdt_stat_slabs_per_image(8, 8) == 2
    assert L.vdt_stat_slabs_per_image(28, 28) == 28 and L.vdt_stat_slabs_per_image(14, 14) == 8
    assert L.vdt_stat_slabs_per_image(7, 7) == 0 and L.vdt_stat_slabs_per_image(4, 4) == 0
    x = torch.zeros(2, 7, 7, 64, device="cuda", dtype=torch.float16)
    w = torch.zeros(64, 64, 3, 3, device="cuda")
    b = torch.zeros(64, device="cuda")
    out = torch.zeros(2, 7, 7, 64, device="cuda")
    st = torch.zeros(64, 16, 2, device="cuda")
    rc = L.vdt_op_conv(_p(x), 2, 7, 7, 64, _p(w), 64, 3, _p(b), None, _p(out), 1, None, _p(st), 4, None)
    assert rc != 0 and b"statistics layout" in L.vdt_last_error()


ATTN_CASES = [(2, 1024, 1, 256), (3, 256, 1, 256), (3, 64, 1, 256), (2, 256, 1, 64), (2, 64, 2, 64), (1, 4096, 1, 64),
              (2, 128, 1, 128),
              # MNIST 28x28 -> 14x14 -> 7x7: N = 784 / 196 / 49, ragged last key tile and query tile
              (2, 784, 1, 256), (3, 196, 1, 256), (3, 49, 1, 256), (2, 196, 2, 64), (3, 16, 1, 64)]


@pytest.mark.parametrize("f16", [1, 0])
@pytest.mark.parametrize("B,N,heads,d", ATTN_CASES)
def test_attention(L, B, N, heads, d, f16):
    g = torch.Generator(device="cuda").manual_seed(N + heads * 3 + d)
    hid = heads * d
    q = torch.randn(B, N, heads, d, device="cuda", generator=g).to(DT[f16])
    k = torch.randn(B, N, heads, d, device="cuda", generator=g).to(DT[f16])
    v = torch.randn(B, N, heads, d, device="cuda", generator=g).to(DT[f16])
    # make the softmax peaky in places so the lazy rescale path (row max jumps by > 2^8) is exercised
    q[:, : N // 2] *= 3.0
    k[:, N // 2:] *= 2.0
    qkv = torch.cat([q.reshape(B * N, hid), k.reshape(B * N, hid), v.reshape(B * N, hid)], dim=1).contiguous()
    out = torch.zeros(B * N, hid, device="cuda", dtype=DT[f16])
    _check(L, L.vdt_op_attention(_p(qkv), _p(out), B, N, heads, d, f16, None))
    torch.cuda.synchronize()
    qd, kd, vd = (z.double().permute(0, 2, 1, 3) for z in (q, k, v))           # B, h, N, d
    w = torch.softmax(qd @ kd.transpose(-1, -2) / math.sqrt(d), dim=-1)
    ref = (w @ vd).permute(0, 2, 1, 3).reshape(B * N, hid)
    assert torch.isfinite(out.float()).all()
    assert _rel(out, ref) <= 1e-2 * EPS[f16], _rel(out, ref)           # P and the output are rounded to 16 bits
    assert (out.double() - ref).abs().max().item() <= 6e-2 * EPS[f16]


@pytest.mark.parametrize("mot,cfg,last", [(3, 1, False), (3, 1, True), (0, 0, False), (1, 0, False), (2, 0, False),
                                          (2, 1, True), (3, 0, False)])
def test_sampler_step(L, mot, cfg, last):
    from oracle.diffusion_ref import _pred_x0
    from v_diffusion_b200 import GaussianDiffusion, get_logsnr_schedule
    T, B, Cc, H = 20, 3, 3, 8
    names = {0: "x0", 1: "eps", 2: "both", 3: "v"}
    diff = GaussianDiffusion(get_logsnr_schedule("cosine"), T, names[mot], "fixed_medium", "snr_trunc", "mse",
                             intp_frac=0.3, w_guide=1.5)
    coefs = diff.step_coefficients(use_ddim=False)
    step = 0 if last else 7
    g = torch.Generator(device="cuda").manual_seed(mot * 10 + cfg)
    rep, Cm = 1 + cfg, (2 * Cc if mot == 2 else Cc)
    mo = torch.randn(B * rep, Cm, H, H, device="cuda", generator=g)
    x = torch.randn(B, Cc, H, H, device="cuda", generator=g)
    z = torch.randn(B, Cc, H, H, device="cuda", generator=g)
    out = torch.zeros_like(x)
    _check(L, L.vdt_op_sampler_step(_p(mo), _p(x), _p(z), _p(out), B, Cc, H * H, cfg, mot, step,
                                    _p(coefs[step].contiguous()), 1.5, None))
    torch.cuda.synchronize()
    row = coefs[step]
    lt = row[11].cuda()
    xin = x.repeat_interleave(rep, dim=0)
    x0 = _pred_x0(xin, mo, lt, names[mot]).clamp(-1, 1)
    mean = x0 if last else row[6].cuda() * xin + row[7].cuda() * x0
    if cfg:
        mean = mean[0::2] + 1.5 * (mean[0::2] - mean[1::2])
    if not last:
        mean = mean + row[8].cuda() * z
    assert (out - mean).abs().max().item() <= 2e-5


@pytest.mark.parametrize("f16", [1, 0])
def test_groupnorm_dropout_mask_statistics(L, f16):
    """norm2 -> act2 -> dropout of a ResidualBlock in .train() mode (unet.py:135, 146): every surviving element equals the
    un-dropped activation / (1 - p), the dropped fraction is p within sampling error, masks repeat for a (seed, layer) pair
    and differ across seeds and layers."""
    B, H, Cc, p = 4, 16, 256, 0.2
    g = torch.Generator(device="cuda").manual_seed(5)
    x = torch.randn(B, H, H, Cc, device="cuda", generator=g) * 1.7 + 0.3
    gamma = torch.rand(Cc, device="cuda", generator=g) + 0.5
    beta = torch.randn(Cc, device="cuda", generator=g) * 0.1

    def run(seed, layer):
        out = torch.zeros(B, H, H, Cc, device="cuda", dtype=DT[f16])
        _check(L, L.vdt_op_groupnorm_dropout(_p(x), Cc, B, H, H, _p(gamma), _p(beta), 1, _p(out), f16, C.c_float(p), seed, layer, None))
        torch.cuda.synchronize()
        return out.float()
    ref = F.silu(F.group_norm(x.permute(0, 3, 1, 2), 32, gamma, beta, 1e-6)).permute(0, 2, 3, 1)
    a = run(11, 3)
    kept = a != 0
    frac = 1.0 - kept.float().mean().item()
    n = a.numel()
    assert abs(frac - p) < 5 * math.sqrt(p * (1 - p) / n) + 1e-3, frac      # (+ the few activations that are exactly 0)
    err = ((a - ref / (1 - p)).abs() * kept).max().item()
    assert err <= 3e-2 * EPS[f16] * 4
    assert torch.equal(a, run(11, 3))
    b, c = run(12, 3), run(11, 4)
    for other in (b, c):
        agree = ((other != 0) == kept).float().mean().item()
        assert abs(agree - (p * p + (1 - p) ** 2)) < 0.01, agree             # independent masks agree with probability p^2 + (1-p)^2
    # every channel and every pixel sees its share of drops (no structure along either axis)
    per_c = 1.0 - kept.float().mean(dim=(0, 1, 2))
    per_px = 1.0 - kept.float().mean(dim=3)
    assert (per_c - p).abs().max().item() < 0.08 and (per_px - p).abs().max().item() < 0.15


GN_BWD_CASES = [
    # B, H, W, C, film, silu, drop_p
    (4, 32, 32, 256, True, 1, 0.0),      # norm2 of the CIFAR network: FiLM + SiLU
    (3, 16, 16, 512, False, 1, 0.0),     # norm1 of a concat block
    (5, 8, 8, 256, True, 1, 0.2),        # training mode: dropout mask regenerated from the forward's stream
    (2, 28, 28, 128, True, 0, 0.0),      # no activation (out_conv-style norm), odd pixel count per slab
    (2, 7, 9, 1024, False, 1, 0.3),
]


@pytest.mark.parametrize("case", GN_BWD_CASES)
def test_groupnorm_backward_vs_autograd(L, case):
    """Backward of GroupNorm(32, 1e-6) -> FiLM -> SiLU -> dropout (unet.py:131-135, 143-146) against fp64 autograd through
    F.group_norm / F.silu with the forward kernel's own dropout mask: grad_x, grad_gamma, grad_beta and the FiLM
    (shift, scale) gradients."""
    B, H, W, Cc, film_on, silu, p = case
    g = torch.Generator(device="cuda").manual_seed(17)
    x = torch.randn(B, H, W, Cc, device="cuda", generator=g) * 1.3 + 0.4
    gamma = torch.rand(Cc, device="cuda", generator=g) + 0.5
    beta = torch.randn(Cc, device="cuda", generator=g) * 0.2
    film = (torch.randn(B, 2 * Cc, device="cuda", generator=g) * 0.3) if film_on else None
    go = torch.randn(B, H, W, Cc, device="cuda", generator=g)
    seed, layer = 1234567, 9
    mask = None
    if p > 0:
        # the forward's mask: the dropout op has no FiLM input, but the mask only depends on (seed, layer, element index)
        out = torch.zeros(B, H, W, Cc, device="cuda", dtype=torch.float16)
        _check(L, L.vdt_op_groupnorm_dropout(_p(x), Cc, B, H, W, _p(gamma), _p(beta), 0, _p(out), 1, C.c_float(p), seed, layer, None))
        torch.cuda.synchronize()
        mask = (out != 0).double() / (1 - p)
    xd = x.double().requires_grad_(True)
    gd, bd = gamma.double().requires_grad_(True), beta.double().requires_grad_(True)
    fd = film.double().requires_grad_(True) if film_on else None
    y = F.group_norm(xd.permute(0, 3, 1, 2), 32, gd, bd, 1e-6).permute(0, 2, 3, 1)
    if film_on:
        y = y * (1 + fd[:, Cc:].view(B, 1, 1, Cc)) + fd[:, :Cc].view(B, 1, 1, Cc)        # unet.py:145: shift first, scale second
    if silu:
        y = F.silu(y)
    if mask is not None:
        y = y * mask
    (y * go.double()).sum().backward()
    gx = torch.empty_like(x)
    gg, gb = torch.empty(Cc, device="cuda"), torch.empty(Cc, device="cuda")
    gf = torch.empty(B, 2 * Cc, device="cuda") if film_on else None
    _check(L, L.vdt_op_groupnorm_backward(_p(x), _p(go), Cc, B, H, W, _p(gamma), _p(beta), _p(film) if film_on else None, silu,
                                          C.c_float(p), seed, layer, _p(gx), _p(gg), _p(gb), _p(gf) if film_on else None, None))
    torch.cuda.synchronize()

    def rel(a, b):
        return ((a.double() - b).norm() / b.norm()).item()
    errs = {"x": rel(gx, xd.grad), "gamma": rel(gg, gd.grad), "beta": rel(gb, bd.grad)}
    if film_on:
        errs["film"] = rel(gf, fd.grad)
    print(f"groupnorm backward {case}: " + ", ".join(f"d{k} {v:.2e}" for k, v in errs.items()))
    assert max(errs.values()) < 2e-5, errs
    gx2 = torch.empty_like(x)
    _check(L, L.vdt_op_groupnorm_backward(_p(x), _p(go), Cc, B, H, W, _p(gamma), _p(beta), _p(film) if film_on else None, silu,
                                          C.c_float(p), seed, layer, _p(gx2), _p(gg), _p(gb), _p(gf) if film_on else None, None))
    torch.cuda.synchronize()
    assert torch.equal(gx, gx2)                                  # fixed-order reductions: bit-reproducible


BWD_CASES = [
    # B, H, cin, cout, k
    (4, 32, 256, 256, 3),       # the dominant shape of the CIFAR network
    (3, 16, 512, 256, 3),       # concat block conv1: two input-channel blocks, odd batch
    (5, 8, 256, 256, 3),        # two images per 128-pixel tile, zero-filled tail
    (2, 32, 512, 256, 1),       # 1x1 skip conv
    (2, 16, 128, 128, 3),
    (2, 64, 192, 384, 3),       # CelebA-style widths (192-wide input-channel block)
]


@pytest.mark.parametrize("f16", [1, 0])
@pytest.mark.parametrize("B,H,cin,cout,k", BWD_CASES)
def test_conv_backward_vs_autograd(L, B, H, cin, cout, k, f16):
    """dgrad and wgrad (+ bias grad) of a conv layer against torch autograd in fp64 on the same 16-bit-rounded operands."""
    g = torch.Generator(device="cuda").manual_seed(H + cin + k)
    x = torch.randn(B, H, H, cin, device="cuda", generator=g).to(DT[f16])
    dy = torch.randn(B, H, H, cout, device="cuda", generator=g).to(DT[f16])
    w = (torch.randn(cout, cin, k, k, device="cuda", generator=g) / math.sqrt(cin * k * k))
    dx = torch.zeros(B, H, H, cin, device="cuda")
    dw = torch.zeros(cout, cin, k, k, device="cuda")
    db = torch.zeros(cout, device="cuda")
    _check(L, L.vdt_op_conv_dgrad(_p(dy), B, H, H, cin, _p(w), cout, k, _p(dx), f16, None))
    _check(L, L.vdt_op_conv_wgrad(_p(x), _p(dy), B, H, H, cin, cout, k, _p(dw), _p(db), f16, None))
    torch.cuda.synchronize()
    xd = x.double().permute(0, 3, 1, 2).requires_grad_(True)
    wd = w.to(DT[f16]).double().requires_grad_(True)           # dgrad multiplies by the 16-bit-rounded weight
    bd = torch.zeros(cout, device="cuda", dtype=torch.float64, requires_grad=True)
    y = F.conv2d(xd, wd, bd, padding=k // 2)
    y.backward(dy.double().permute(0, 3, 1, 2))
    ref_dx = xd.grad.permute(0, 2, 3, 1)
    print(f"conv backward {cin}->{cout} k{k} @{H}: dgrad rel {_rel(dx, ref_dx):.2e} wgrad rel {_rel(dw, wd.grad):.2e} dbias rel {_rel(db, bd.grad):.2e}")
    assert _rel(dx, ref_dx) <= 2e-3 * EPS[f16] + 1e-5        # fp32 accumulation of exact 16-bit products
    assert _rel(dw, wd.grad) <= 1e-4
    assert _rel(db, bd.grad) <= 1e-5
    # deterministic: fixed-order split reduction
    dw2 = torch.zeros_like(dw)
    _check(L, L.vdt_op_conv_wgrad(_p(x), _p(dy), B, H, H, cin, cout, k, _p(dw2), None, f16, None))
    torch.cuda.synchronize()
    assert torch.equal(dw, dw2)


@pytest.mark.parametrize("f16", [1, 0])
@pytest.mark.parametrize("B,H,Cc", [(4, 16, 256), (2, 32, 256)])
def test_residual_block_backward_composed_from_kernels(L, B, H, Cc, f16):
    """A 256 -> 256 ResidualBlock (unet.py:106-148, eval-mode dropout) forward and backward, composed from this library's
    kernels only -- GroupNorm fwd / bwd, conv fwd / dgrad / wgrad -- against fp64 autograd of the same block: the output,
    d x, every parameter gradient and the FiLM (t_emb projection) gradient.  16-bit operands round activations, weights and
    the gradients fed to dgrad / wgrad; everything else is fp32."""
    g = torch.Generator(device="cuda").manual_seed(31 + H)
    x = torch.randn(B, H, H, Cc, device="cuda", generator=g) * 1.2
    film = torch.randn(B, 2 * Cc, device="cuda", generator=g) * 0.3
    go = torch.randn(B, H, H, Cc, device="cuda", generator=g)
    P = {}
    for i in (1, 2):
        P[f"g{i}"] = torch.rand(Cc, device="cuda", generator=g) + 0.5
        P[f"be{i}"] = torch.randn(Cc, device="cuda", generator=g) * 0.2
        P[f"w{i}"] = torch.randn(Cc, Cc, 3, 3, device="cuda", generator=g) / math.sqrt(Cc * 9)
        P[f"b{i}"] = torch.randn(Cc, device="cuda", generator=g) * 0.1
    dt = DT[f16]

    def gn(src, gamma, beta, ftab):
        out = torch.empty(B, H, H, Cc, device="cuda", dtype=dt)
        _check(L, L.vdt_op_groupnorm(_p(src), Cc, None, 0, B, H, H, _p(gamma), _p(beta), _p(ftab), 2 * Cc, 0, 1, 0, _p(out), None, None,
                                     f16, None, None, 4, 0, None))
        return out

    def conv(a, w, b, resid):
        out = torch.empty(B, H, H, Cc, device="cuda")
        _check(L, L.vdt_op_conv(_p(a), B, H, H, Cc, _p(w), Cc, 3, _p(b), _p(resid), _p(out), f16, None, None, 4, None))
        return out

    def conv_bwd(a, dy, w):
        dy16 = dy.to(dt)
        dx, dw, db = torch.empty(B, H, H, Cc, device="cuda"), torch.empty_like(w), torch.empty(Cc, device="cuda")
        _check(L, L.vdt_op_conv_dgrad(_p(dy16), B, H, H, Cc, _p(w), Cc, 3, _p(dx), f16, None))
        _check(L, L.vdt_op_conv_wgrad(_p(a), _p(dy16), B, H, H, Cc, Cc, 3, _p(dw), _p(db), f16, None))
        return dx, dw, db

    def gn_bwd(src, dy, gamma, beta, ftab):
        dx, dg, db = torch.empty_like(src), torch.empty(Cc, device="cuda"), torch.empty(Cc, device="cuda")
        df = torch.empty_like(ftab) if ftab is not None else None
        _check(L, L.vdt_op_groupnorm_backward(_p(src), _p(dy), Cc, B, H, H, _p(gamma), _p(beta), _p(ftab), 1, C.c_float(0.0), 0, 0,
                                              _p(dx), _p(dg), _p(db), _p(df), None))
        return dx, dg, db, df
    # forward
    a1 = gn(x, P["g1"], P["be1"], None)
    h1 = conv(a1, P["w1"], P["b1"], None)
    a2 = gn(h1, P["g2"], P["be2"], film)
    out = conv(a2, P["w2"], P["b2"], x)
    # backward
    got = {}
    da2, got["w2"], got["b2"] = conv_bwd(a2, go, P["w2"])
    dh1, got["g2"], got["be2"], got["film"] = gn_bwd(h1, da2, P["g2"], P["be2"], film)
    da1, got["w1"], got["b1"] = conv_bwd(a1, dh1, P["w1"])
    dxg, got["g1"], got["be1"], _ = gn_bwd(x, da1, P["g1"], P["be1"], None)
    got["x"] = dxg + go                                           # identity skip
    torch.cuda.synchronize()
    # fp64 autograd of the same block
    R = {k: v.double().requires_grad_(True) for k, v in P.items()}
    xd, fd = x.double().requires_grad_(True), film.double().requires_grad_(True)
    nchw = lambda t: t.permute(0, 3, 1, 2)
    y = F.silu(F.group_norm(nchw(xd), 32, R["g1"], R["be1"], 1e-6))
    y = F.conv2d(y, R["w1"], R["b1"], padding=1)
    y = F.group_norm(y, 32, R["g2"], R["be2"], 1e-6)
    y = F.silu(y * (1 + fd[:, Cc:].view(B, Cc, 1, 1)) + fd[:, :Cc].view(B, Cc, 1, 1))
    y = F.conv2d(y, R["w2"], R["b2"], padding=1) + nchw(xd)
    y.backward(nchw(go.double()))
    want = {k: v.grad for k, v in R.items()}
    want["x"], want["film"] = xd.grad, fd.grad
    errs = {"out": _rel(out, y.detach().permute(0, 2, 3, 1))}
    errs.update({"d" + k: _rel(got[k], want[k]) for k in sorted(got)})
    print(f"ResidualBlock fwd+bwd {Cc}ch @{H} B={B} {'fp16' if f16 else 'bf16'}: " + ", ".join(f"{k} {v:.1e}" for k, v in errs.items()))
    assert max(errs.values()) <= 8e-3 * EPS[f16], errs          # measured: 5.6e-4 (fp16), 4.3e-3 (bf16)


@pytest.mark.parametrize("B,N,heads,d", [(2, 64, 1, 256), (3, 256, 4, 64), (1, 100, 2, 128), (1, 1024, 1, 256), (2, 49, 3, 192)])
def test_attn_core_backward_vs_autograd(L, B, N, heads, d):
    """dQ, dK, dV of softmax(q k^T / sqrt(d)) v (unet.py:55-64) from the fp32 two-pass backward against fp64 autograd."""
    g = torch.Generator(device="cuda").manual_seed(N + heads + d)
    hid = heads * d
    qkv = torch.randn(B * N, 3 * hid, device="cuda", generator=g)
    qkv[:, :hid] *= 1.5                                           # some peaky rows
    go = torch.randn(B * N, hid, device="cuda", generator=g)
    dqkv = torch.zeros_like(qkv)
    _check(L, L.vdt_op_attention_backward(_p(qkv), _p(go), _p(dqkv), B, N, heads, d, None))
    torch.cuda.synchronize()
    x = qkv.double().requires_grad_(True)
    q, k, v = (x[:, i * hid:(i + 1) * hid].reshape(B, N, heads, d).permute(0, 2, 1, 3) for i in range(3))
    w = torch.softmax(q @ k.transpose(-1, -2) / math.sqrt(d), dim=-1)
    out = (w @ v).permute(0, 2, 1, 3).reshape(B * N, hid)
    out.backward(go.double())
    errs = [_rel(dqkv[:, i * hid:(i + 1) * hid], x.grad[:, i * hid:(i + 1) * hid]) for i in range(3)]
    print(f"attention backward B={B} N={N} heads={heads} d={d}: dq {errs[0]:.1e} dk {errs[1]:.1e} dv {errs[2]:.1e}")
    assert max(errs) <= 2e-5
    again = torch.zeros_like(qkv)
    _check(L, L.vdt_op_attention_backward(_p(qkv), _p(go), _p(again), B, N, heads, d, None))
    torch.cuda.synchronize()
    assert torch.equal(dqkv, again)


@pytest.mark.parametrize("f16", [1, 0])
def test_attn_block_backward_composed_from_kernels(L, f16):
    """An AttentionBlock (unet.py:33-81: GroupNorm -> 1x1 proj_in -> softmax(q k^T / sqrt(d)) v -> 1x1 proj_out -> + x) forward
    and backward composed from this library's kernels only, against fp64 autograd: output, d x and every parameter gradient.
    Forward on the tensor-core kernels (16-bit q | k | v and output); the core's backward is the fp32 reference-grade kernel."""
    B, H, Cc, heads = 3, 16, 256, 1
    N, d, hid = H * H, 256, 256
    dt = DT[f16]
    g = torch.Generator(device="cuda").manual_seed(41)
    x = torch.randn(B, H, H, Cc, device="cuda", generator=g) * 1.1
    go = torch.randn(B, H, H, Cc, device="cuda", generator=g)
    P = {"g": torch.rand(Cc, device="cuda", generator=g) + 0.5, "be": torch.randn(Cc, device="cuda", generator=g) * 0.2,
         "w_in": torch.randn(3 * hid, Cc, 1, 1, device="cuda", generator=g) / math.sqrt(Cc), "b_in": torch.randn(3 * hid, device="cuda", generator=g) * 0.1,
         "w_out": torch.randn(Cc, hid, 1, 1, device="cuda", generator=g) / math.sqrt(hid), "b_out": torch.randn(Cc, device="cuda", generator=g) * 0.1}
    # forward
    a = torch.empty(B, H, H, Cc, device="cuda", dtype=dt)
    _check(L, L.vdt_op_groupnorm(_p(x), Cc, None, 0, B, H, H, _p(P["g"]), _p(P["be"]), None, 0, 0, 0, 0, _p(a), None, None, f16, None, None,
                                 4, 0, None))
    qkv32 = torch.empty(B, H, H, 3 * hid, device="cuda")
    qkv16 = torch.empty(B, H, H, 3 * hid, device="cuda", dtype=dt)
    _check(L, L.vdt_op_conv(_p(a), B, H, H, Cc, _p(P["w_in"]), 3 * hid, 1, _p(P["b_in"]), None, _p(qkv32), f16, _p(qkv16), None, 4, None))
    o16 = torch.empty(B * N, hid, device="cuda", dtype=dt)
    _check(L, L.vdt_op_attention(_p(qkv16), _p(o16), B, N, heads, d, f16, None))
    out = torch.empty(B, H, H, Cc, device="cuda")
    _check(L, L.vdt_op_conv(_p(o16), B, H, H, hid, _p(P["w_out"]), Cc, 1, _p(P["b_out"]), _p(x), _p(out), f16, None, None, 4, None))
    # backward
    got = {}
    go16 = go.to(dt)
    do = torch.empty(B, H, H, hid, device="cuda")
    got["w_out"], got["b_out"] = torch.empty_like(P["w_out"]), torch.empty(Cc, device="cuda")
    _check(L, L.vdt_op_conv_dgrad(_p(go16), B, H, H, hid, _p(P["w_out"]), Cc, 1, _p(do), f16, None))
    _check(L, L.vdt_op_conv_wgrad(_p(o16), _p(go16), B, H, H, hid, Cc, 1, _p(got["w_out"]), _p(got["b_out"]), f16, None))
    dqkv = torch.empty(B * N, 3 * hid, device="cuda")
    qkvf = qkv16.float().reshape(B * N, 3 * hid).contiguous()
    _check(L, L.vdt_op_attention_backward(_p(qkvf), _p(do), _p(dqkv), B, N, heads, d, None))
    dqkv16 = dqkv.to(dt)
    da = torch.empty(B, H, H, Cc, device="cuda")
    got["w_in"], got["b_in"] = torch.empty_like(P["w_in"]), torch.empty(3 * hid, device="cuda")
    _check(L, L.vdt_op_conv_dgrad(_p(dqkv16), B, H, H, Cc, _p(P["w_in"]), 3 * hid, 1, _p(da), f16, None))
    _check(L, L.vdt_op_conv_wgrad(_p(a), _p(dqkv16), B, H, H, Cc, 3 * hid, 1, _p(got["w_in"]), _p(got["b_in"]), f16, None))
    dx, got["g"], got["be"] = torch.empty_like(x), torch.empty(Cc, device="cuda"), torch.empty(Cc, device="cuda")
    _check(L, L.vdt_op_groupnorm_backward(_p(x), _p(da), Cc, B, H, H, _p(P["g"]), _p(P["be"]), None, 0, C.c_float(0.0), 0, 0,
                                          _p(dx), _p(got["g"]), _p(got["be"]), None, None))
    got["x"] = dx + go
    torch.cuda.synchronize()
    # fp64 autograd of the same block
    R = {k: v.double().requires_grad_(True) for k, v in P.items()}
    xd = x.double().requires_grad_(True)
    y = F.group_norm(xd.permute(0, 3, 1, 2), 32, R["g"], R["be"], 1e-6)
    qkv = F.conv2d(y, R["w_in"], R["b_in"]).permute(0, 2, 3, 1).reshape(B, N, 3 * hid)
    q, k, v = (qkv[..., i * hid:(i + 1) * hid].reshape(B, N, heads, d).permute(0, 2, 1, 3) for i in range(3))
    o = (torch.softmax(q @ k.transpose(-1, -2) / math.sqrt(d), dim=-1) @ v).permute(0, 2, 1, 3).reshape(B, H, H, hid)
    yo = F.conv2d(o.permute(0, 3, 1, 2), R["w_out"], R["b_out"]) + xd.permute(0, 3, 1, 2)
    yo.backward(go.double().permute(0, 3, 1, 2))
    want = {k: v.grad for k, v in R.items()}
    want["x"] = xd.grad
    errs = {"out": _rel(out, yo.detach().permute(0, 2, 3, 1))}
    errs.update({"d" + k: _rel(got[k], want[k]) for k in sorted(got)})
    print(f"AttentionBlock fwd+bwd {Cc}ch N={N} B={B} {'fp16' if f16 else 'bf16'}: " + ", ".join(f"{k} {v:.1e}" for k, v in errs.items()))
    assert max(errs.values()) <= 8e-3 * EPS[f16], errs          # measured: 7.7e-4 (fp16), 5.8e-3 (bf16)

