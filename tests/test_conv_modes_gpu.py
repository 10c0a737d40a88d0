"""GPU parity of the conv modes only the sampler's plan reaches, one launch at a time (vdt_op_conv_ex, vdt_op_in_conv,
vdt_op_out_conv): the sub-pixel 2x-upsampling conv, the upsampled and the pair-shared residual, the fused 1x1 skip conv,
the split-precision segments, in_conv and out_conv.  Each case compares against fp64 torch of the same operation on the
same 16-bit-rounded operands, at the map sizes where the conv kernel changes epilogue (fast power-of-two remaps, the
generic epilogue of 28 / 14 / 7 / 4 and of ragged tiles), and checks the GroupNorm statistics the epilogue writes both
directly and through the single-pass GroupNorm that consumes them.

Epilogue variants of conv_gemm.cu and the cases that reach them (with all 32 rows of a quarter valid; ragged quarters
always take the generic epilogue):
  0-2   fp32 out + residual, stats 4 / 2 / none   test_resid_rep_bit_identical (the materialised mode-0 run at 16, 32)
  3-5   fp32 out                                  test_conv_skip at 32, 16, 8
  6-8   16-bit out                                test_conv_skip at 32, 16 (out16); test_fp16_saturation "plain"
  9-11  ups, fp32 out                             test_ups at 8, 16, 32 (low-res side)
  12-14 ups, 16-bit out                           test_ups at 8, 16, 32 with out16
  15-17 resid_up, fp32 out                        test_resid_up at 8, 16, 32, 64
  18-20 resid_rep = 2, fp32 out                   test_resid_rep_bit_identical at 8, 16, 32
  generic                                         maps 28 / 14 / 7 / 4 of every mode, 16-bit out with a residual,
                                                  the ragged last tile of the ups case at 8 with an odd batch
"""
import ctypes as C
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DT = {1: torch.float16, 0: torch.bfloat16}
U16 = {1: 2.0 ** -11, 0: 2.0 ** -8}          # unit roundoff of the 16-bit formats
EPS = {1: 0.25, 0: 1.0}                      # rounding unit relative to bf16 (as in test_gpu_kernels)
FMT = {1: "fp16", 0: "bf16"}

# Bars, each about 2-5x the worst value measured over every case of this file on a B200 at its 1000 W power limit
# (profiles/r7_conv_modes_parity.txt)
ACC_ABS = 1e-4        # max |out - ref| of fp32 outputs, fp32 accumulation of exact 16-bit products: measured 2.1e-5 (skip, 32)
ACC_16 = 5e-5         # 16-bit outputs: |out - ref| <= u |ref| + ACC_16; measured 1.0e-5 (skip, 32, fp16)
UPS_LOOSE = 6.0       # ups against conv(upsample(x), round16(w)): max |err| / (u * sqrt(conv(U^2, W^2))), a bound in
                      # standard deviations of the weight rounding; measured 2.9 (fp16 and bf16)
STAT_REL = 4e-5       # |sum - ref| / sum |v|, |sumsq - ref| / sum v^2, per slab and per image: measured 1.1e-5 (split, 16)
SPLIT_REL = 2e-5      # split-precision (fp16x3) rel-L2 against fp64 on the fp32 operands: measured 5.0e-6


@pytest.fixture(scope="module")
def L():
    from v_diffusion_b200 import _lib
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return _lib.lib()


def _addr(t):
    return None if t is None else t.data_ptr()


def _check(L, rc):
    assert rc == 0, L.vdt_last_error().decode()


def _rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


def _conv_ex(L, *, a3, w3, bias, c3, cout, batch, h, w, f16, a3_lo=None, a1=None, a1_lo=None, w1=None, c1=0, residual=None,
             resid_mode=0, ups=0, out16=False, sc=0, sat=None):
    """One vdt_op_conv_ex call; returns (output, statistics or None)."""
    from v_diffusion_b200 import _lib
    H, W = (2 * h, 2 * w) if ups else (h, w)
    out = torch.full((batch, H, W, cout), float("nan"), device="cuda", dtype=DT[f16] if out16 else torch.float32)
    stats = None
    if sc:
        slabs = L.vdt_stat_slabs_per_image(H, W)
        stats = torch.full((batch * slabs + 4, cout // sc, 2), float("nan"), device="cuda")
    op = _lib.ConvOp(a3=_addr(a3), a3_lo=_addr(a3_lo), a1=_addr(a1), a1_lo=_addr(a1_lo), w3=_addr(w3), w1=_addr(w1),
                     bias=_addr(bias), residual=_addr(residual), out_f32=None if out16 else _addr(out),
                     out16=_addr(out) if out16 else None, stats=_addr(stats), sat_count=_addr(sat), batch=batch, h=h, w=w,
                     c3=c3, c1=c1, cout=cout, ups=ups, resid_mode=resid_mode, stat_cols=sc or 4, f16=f16)
    _check(L, L.vdt_op_conv_ex(C.byref(op), None))
    torch.cuda.synchronize()
    return out, stats


def _nhwc(t):
    return t.permute(0, 2, 3, 1)


def _nchw(t):
    return t.permute(0, 3, 1, 2)


def _weights(g, cout, cin, k=3):
    return torch.randn(cout, cin, k, k, device="cuda", generator=g) / math.sqrt(cin * k * k)


def _act(g, B, h, w, c, f16, scale=1.0):
    return (torch.randn(B, h, w, c, device="cuda", generator=g) * scale).to(DT[f16])


def _check_out(out, ref, f16, tag):
    """fp32 output: max-abs bar; 16-bit output: within the format's rounding of the exact value."""
    assert torch.isfinite(out.float()).all(), tag
    d = (out.double() - ref).abs()
    if out.dtype == torch.float32:
        err = d.max().item()
        print(f"PARITY {tag} out_f32 maxabs {err:.3e}")
        assert err <= ACC_ABS, f"{tag}: max abs err {err}"
    else:
        err = (d - U16[f16] * ref.abs()).max().item()
        print(f"PARITY {tag} out16 excess {err:.3e}")
        assert err <= ACC_16, f"{tag}: 16-bit err beyond rounding {err}"


def _check_stats(L, stats, ref, B, sc, tag, parity_low=None):
    """Statistics rows [0, B * slabs) are finite; per image they add up to the reference's sum / sum of squares per column
    group; where every slab is 32 consecutive rows, each slab matches too.  parity_low = (h, w): a sub-pixel conv output,
    whose slab (img * 4 + par) * slabs(h, w) + s holds low-resolution rows [32 s, 32 s + 32) of parity class par."""
    H, W, cout = ref.shape[1], ref.shape[2], ref.shape[3]
    slabs = L.vdt_stat_slabs_per_image(H, W)
    st = stats[:B * slabs].double()
    assert torch.isfinite(st).all(), tag
    ri = ref.reshape(B, H * W, cout // sc, sc)
    tot = st.reshape(B, slabs, cout // sc, 2).sum(dim=1)
    e_sum = ((tot[..., 0] - ri.sum(dim=(1, 3))).abs() / ri.abs().sum(dim=(1, 3))).max().item()
    e_sq = ((tot[..., 1] - (ri * ri).sum(dim=(1, 3))).abs() / (ri * ri).sum(dim=(1, 3))).max().item()
    print(f"PARITY {tag} stats_image rel {max(e_sum, e_sq):.3e}")
    assert max(e_sum, e_sq) <= STAT_REL, (tag, e_sum, e_sq)
    h, w = parity_low if parity_low else (H, W)
    if (h * w) % 128 == 0 or 2 * h * w <= 128:             # whole tiles: a slab is 32 consecutive (low-res) rows
        if parity_low:
            want = torch.stack([ref[:, py::2, px::2, :] for py in (0, 1) for px in (0, 1)], dim=1)   # B, par, h, w, cout
        else:
            want = ref[:, None]
        rs = want.reshape(-1, 32, cout // sc, sc)
        ws, wq = rs.sum(dim=(1, 3)), (rs * rs).sum(dim=(1, 3))
        e1 = ((st[..., 0] - ws).abs() / rs.abs().sum(dim=(1, 3))).max().item()
        e2 = ((st[..., 1] - wq).abs() / wq).max().item()
        print(f"PARITY {tag} stats_slab rel {max(e1, e2):.3e}")
        assert max(e1, e2) <= STAT_REL, (tag, e1, e2)


def _check_groupnorm(L, out, stats, ref, B, sc, f16, tag):
    """The slabs feed the single-pass GroupNorm at the output resolution (in16 for a 16-bit output), against F.group_norm."""
    H, W, cout = ref.shape[1], ref.shape[2], ref.shape[3]
    g = torch.Generator(device="cuda").manual_seed(H + cout)
    gamma = 1 + 0.2 * torch.randn(cout, device="cuda", generator=g)
    beta = 0.2 * torch.randn(cout, device="cuda", generator=g)
    act = torch.zeros(B, H, W, cout, device="cuda", dtype=DT[f16])
    in16 = int(out.dtype != torch.float32)
    _check(L, L.vdt_op_groupnorm(C.c_void_p(out.data_ptr()), cout, None, 0, B, H, W, C.c_void_p(gamma.data_ptr()),
                                 C.c_void_p(beta.data_ptr()), None, 0, 0, 1, 0, C.c_void_p(act.data_ptr()), None, None, f16,
                                 C.c_void_p(stats.data_ptr()), None, sc, in16, None))
    torch.cuda.synchronize()
    x = out.double() if in16 else ref                       # the kernel normalises the rounded values with fp32 statistics
    y = _nhwc(F.silu(F.group_norm(_nchw(x), 32, gamma.double(), beta.double(), 1e-6)))
    rel = _rel(act, y)
    print(f"PARITY {tag} groupnorm rel {rel:.3e}")
    assert rel <= 4e-3 * EPS[f16] + (2e-3 if in16 else 0), (tag, rel)


def _outputs(cout, stats_ok):
    """(out16, stat_cols) combinations: fp32 / 16-bit output x statistics none / 4 / 2 where the layout exists and the
    GroupNorm can consume it (columns per entry divide the 32 groups' channel count)."""
    combos = [(False, 0), (True, 0)]
    if stats_ok:
        scs = [s for s in (4, 2) if (cout // 32) % s == 0]
        combos += [(False, s) for s in scs] + [(True, scs[0])]
    return combos


# ---------------------------------------------------------------------------------------------------- sub-pixel conv
def _ups_weights_presummed(w, f16):
    """pack_conv_ups_kernel restated: for parity (py, px) the 3x3 taps reading the same low-res pixel, summed in fp32 in
    the kernel's r, c order, rounded to 16 bits -> [4 parities][cout, cin, 2, 2] (tap (ty, tx) reads low-res pixel
    (y + ty - 1 + py, x + tx - 1 + px))."""
    out = []
    for py in (0, 1):
        for px in (0, 1):
            k = torch.zeros(w.shape[0], w.shape[1], 2, 2, device=w.device)
            for ty in (0, 1):
                for tx in (0, 1):
                    s = None
                    for r in range(3):
                        if (py + r - 1) // 2 + 1 - py != ty:
                            continue
                        for c in range(3):
                            if (px + c - 1) // 2 + 1 - px != tx:
                                continue
                            s = w[:, :, r, c].clone() if s is None else s + w[:, :, r, c]
                    k[:, :, ty, tx] = s
            out.append(k.to(DT[f16]).double())
    return out


def _ups_ref_subpixel(x16, w, bias, f16):
    B, h, w_, _ = x16.shape
    xp = F.pad(_nchw(x16.double()), (1, 1, 1, 1))
    ks = _ups_weights_presummed(w, f16)
    out = torch.zeros(B, w.shape[0], 2 * h, 2 * w_, device="cuda", dtype=torch.float64)
    for par, k in enumerate(ks):
        py, px = par >> 1, par & 1
        out[:, :, py::2, px::2] = F.conv2d(xp[:, :, py:py + h + 1, px:px + w_ + 1], k)
    return _nhwc(out + bias.double()[None, :, None, None])


UPS_CASES = [
    # B, h (low-res side), c (= cin = cout)
    (3, 8, 128),      # 8 -> 16: two images per tile (fast MAP 1), odd batch -> ragged last tile (generic, phantom image)
    (2, 16, 256),     # 16 -> 32
    (1, 32, 192),     # 32 -> 64 (CelebA width)
    (3, 7, 128),      # 7 -> 14: 98-row tiles of two images, odd batch: generic scatter, no statistics layout
    (2, 14, 128),     # 14 -> 28: generic scatter; 4 * slabs(14) != slabs(28): no statistics
    (2, 4, 64),       # 4 -> 8: eight images per tile, generic scatter
]


def _ups_params():
    out = []
    for B, h, c in UPS_CASES:
        stats_ok = h in (8, 16, 32)          # 4 * slabs(h, h) == slabs(2h, 2h) (test_conv_modes_cpu checks the others refuse)
        for f16 in (1, 0):
            for out16, sc in _outputs(c, stats_ok):
                out.append((B, h, c, f16, out16, sc))
    return out


@pytest.mark.parametrize("B,h,c,f16,out16,sc", _ups_params())
def test_ups(L, B, h, c, f16, out16, sc):
    """Sub-pixel 2x-upsampling conv (conv1 of an upsampling block): tight against the restated sub-pixel form, loose against
    the plain conv of the nearest-upsampled input, which pins the parity / tap rule independently of the restatement."""
    g = torch.Generator(device="cuda").manual_seed(100 * h + c + B)
    x = _act(g, B, h, h, c, f16)
    w = _weights(g, c, c)
    bias = torch.randn(c, device="cuda", generator=g) * 0.5
    out, stats = _conv_ex(L, a3=x, w3=w, bias=bias, c3=c, cout=c, batch=B, h=h, w=h, f16=f16, ups=1, out16=out16, sc=sc)
    tag = f"ups {h}->{2 * h} B{B} c{c} {FMT[f16]} {'out16' if out16 else 'f32'} sc{sc}"
    ref = _ups_ref_subpixel(x, w, bias, f16)
    _check_out(out, ref, f16, tag)
    # loose: the plain definition with the 3x3 weights rounded one by one
    U = F.interpolate(_nchw(x.double()), scale_factor=2, mode="nearest")
    plain = _nhwc(F.conv2d(U, w.to(DT[f16]).double(), bias.double(), padding=1))
    sigma = _nhwc(F.conv2d(U * U, w.double() ** 2, padding=1).sqrt())
    ratio = ((ref - plain).abs() / (U16[f16] * sigma + 1e-30)).max().item()   # what rounding the pre-summed weights moved
    err = (out.double() - plain).abs()
    if out16:
        err = err - U16[f16] * plain.abs()
    ratio_out = (err / (U16[f16] * sigma + 1e-30)).max().item()
    print(f"PARITY {tag} ups_loose ratio {ratio_out:.3e} (presum rounding alone {ratio:.3e})")
    assert ratio_out <= UPS_LOOSE, (tag, ratio_out)
    if sc:
        _check_stats(L, stats, ref, B, sc, tag, parity_low=(h, h))
        _check_groupnorm(L, out, stats, ref, B, sc, f16, tag)


# ---------------------------------------------------------------------------------------------------- resid_up
RESID_UP_CASES = [
    # B, H (output side), c
    (2, 16, 128), (2, 32, 256), (1, 64, 192), (3, 8, 128),     # fast MAP 2 (box_n = 2 at 8, odd batch)
    (3, 14, 128), (2, 28, 64),                                 # generic
]


def _resid_up_params():
    out = []
    for B, H, c in RESID_UP_CASES:
        for f16 in (1, 0):
            for out16, sc in _outputs(c, True):
                out.append((B, H, c, f16, out16, sc))
    return out


@pytest.mark.parametrize("B,H,c,f16,out16,sc", _resid_up_params())
def test_resid_up(L, B, H, c, f16, out16, sc):
    """conv2 of an upsampling block: the identity-skip residual is the low-resolution stream, nearest-upsampled."""
    g = torch.Generator(device="cuda").manual_seed(200 * H + c + B)
    x = _act(g, B, H, H, c, f16)
    w = _weights(g, c, c)
    bias = torch.randn(c, device="cuda", generator=g) * 0.5
    res = torch.randn(B, H // 2, H // 2, c, device="cuda", generator=g)
    out, stats = _conv_ex(L, a3=x, w3=w, bias=bias, c3=c, cout=c, batch=B, h=H, w=H, f16=f16, residual=res, resid_mode=1,
                          out16=out16, sc=sc)
    tag = f"resid_up {H} B{B} c{c} {FMT[f16]} {'out16' if out16 else 'f32'} sc{sc}"
    ref = _nhwc(F.conv2d(_nchw(x.double()), w.to(DT[f16]).double(), bias.double(), padding=1)
                + F.interpolate(_nchw(res.double()), scale_factor=2, mode="nearest"))
    _check_out(out, ref, f16, tag)
    if sc:
        _check_stats(L, stats, ref, B, sc, tag)
        _check_groupnorm(L, out, stats, ref, B, sc, f16, tag)


# ---------------------------------------------------------------------------------------------------- resid_rep
RESID_REP_CASES = [
    # B (rows), H, c
    (2, 16, 64), (4, 16, 128), (6, 16, 64), (2, 32, 256), (4, 32, 128), (6, 32, 64),   # fast MAP 3 with pair_tiles
    (4, 28, 64),                                                                        # generic, pair_tiles = 7
    (4, 8, 128),                                                                        # box_n = 2, no pair tiles
]


def _resid_rep_params():
    out = []
    for B, H, c in RESID_REP_CASES:
        for f16 in (1, 0):
            for out16, sc in _outputs(c, True):
                out.append((B, H, c, f16, out16, sc))
    return out


@pytest.mark.parametrize("B,H,c,f16,out16,sc", _resid_rep_params())
def test_resid_rep_bit_identical(L, B, H, c, f16, out16, sc, monkeypatch):
    """conv2 of block 0 under CFG: output image i adds residual image i / 2.  Against fp64, and bit for bit against the
    same call with the residual materialised by repeat_interleave(2) and against the same call without pair tiles: the
    arithmetic and the K order are the same in all three."""
    g = torch.Generator(device="cuda").manual_seed(300 * H + c + B)
    x = _act(g, B, H, H, c, f16)
    w = _weights(g, c, c)
    bias = torch.randn(c, device="cuda", generator=g) * 0.5
    res = torch.randn(B // 2, H, H, c, device="cuda", generator=g)
    kw = dict(a3=x, w3=w, bias=bias, c3=c, cout=c, batch=B, h=H, w=H, f16=f16, out16=out16, sc=sc)
    out, stats = _conv_ex(L, residual=res, resid_mode=2, **kw)
    tag = f"resid_rep {H} B{B} c{c} {FMT[f16]} {'out16' if out16 else 'f32'} sc{sc}"
    ref = _nhwc(F.conv2d(_nchw(x.double()), w.to(DT[f16]).double(), bias.double(), padding=1)) + res.double().repeat_interleave(2, dim=0)
    _check_out(out, ref, f16, tag)
    full, full_stats = _conv_ex(L, residual=res.repeat_interleave(2, dim=0).contiguous(), resid_mode=0, **kw)
    assert torch.equal(out, full), tag
    monkeypatch.setenv("VDT_PAIR_TILES", "0")
    nopair, nopair_stats = _conv_ex(L, residual=res, resid_mode=2, **kw)
    assert torch.equal(out, nopair), tag
    if sc:
        rows = B * L.vdt_stat_slabs_per_image(H, H)         # (the slack rows after them stay NaN)
        assert torch.equal(stats[:rows], nopair_stats[:rows]), tag
        # the mode-0 run may take another epilogue for some quarters (fast vs generic at 28), which orders the four-column
        # sums differently; two-column entries are summed in the same order everywhere
        if sc == 2 or H != 28:
            assert torch.equal(stats[:rows], full_stats[:rows]), tag
        _check_stats(L, stats, ref, B, sc, tag)
        _check_groupnorm(L, out, stats, ref, B, sc, f16, tag)


# ---------------------------------------------------------------------------------------------------- fused 1x1 skip conv
SKIP_CASES = [
    # B, H, c1 (block input = skip operand), c3 = cout
    (2, 32, 512, 256),    # CIFAR concat block
    (2, 16, 384, 192),    # CelebA-width concat block
    (3, 8, 64, 128),      # small network's downward widening block, two images per tile, odd batch
    (3, 28, 128, 64),     # MNIST-style concat block: 112-row tiles
    (3, 14, 64, 128),     # 98-row tiles
    (3, 7, 256, 128),     # two 49-pixel images per tile, odd batch; no statistics layout
]


def _skip_params():
    out = []
    for B, H, c1, c in SKIP_CASES:
        for f16 in (1, 0):
            for out16, sc in _outputs(c, H != 7):
                out.append((B, H, c1, c, f16, out16, sc))
    return out


@pytest.mark.parametrize("B,H,c1,c,f16,out16,sc", _skip_params())
def test_conv_skip(L, B, H, c1, c, f16, out16, sc):
    """conv2 of a widening block: the 3x3 body and the 1x1 skip conv as two K segments of one GEMM (skip weights packed at
    column 9 * cout), one bias."""
    g = torch.Generator(device="cuda").manual_seed(400 * H + c1 + c + B)
    a3 = _act(g, B, H, H, c, f16)
    a1 = _act(g, B, H, H, c1, f16, scale=2.0)
    w3, w1 = _weights(g, c, c), _weights(g, c, c1, 1)
    bias = torch.randn(c, device="cuda", generator=g) * 0.5
    out, stats = _conv_ex(L, a3=a3, w3=w3, bias=bias, c3=c, cout=c, batch=B, h=H, w=H, f16=f16, a1=a1, w1=w1, c1=c1,
                          out16=out16, sc=sc)
    tag = f"skip {H} B{B} c1 {c1} c{c} {FMT[f16]} {'out16' if out16 else 'f32'} sc{sc}"
    ref = _nhwc(F.conv2d(_nchw(a3.double()), w3.to(DT[f16]).double(), bias.double(), padding=1)
                + F.conv2d(_nchw(a1.double()), w1.to(DT[f16]).double()))
    _check_out(out, ref, f16, tag)
    if sc:
        _check_stats(L, stats, ref, B, sc, tag)
        _check_groupnorm(L, out, stats, ref, B, sc, f16, tag)


# ---------------------------------------------------------------------------------------------------- split precision
def _split(x):
    hi = x.to(torch.float16)
    return hi, (x - hi.float()).to(torch.float16)


SPLIT_CASES = [
    # name, B, h, c3, c1, cout, ups, sc
    ("3x3", 2, 16, 128, 0, 128, 0, 4),
    ("3x3", 3, 28, 64, 0, 64, 0, 2),
    ("3x3+skip", 2, 16, 64, 192, 128, 0, 4),       # six K segments: kConvMaxSegs
    ("3x3+skip", 3, 14, 128, 64, 64, 0, 2),
    ("ups", 3, 8, 128, 0, 128, 1, 4),
    ("ups", 2, 7, 64, 0, 64, 1, 0),
]


@pytest.mark.parametrize("name,B,h,c3,c1,cout,ups,sc", SPLIT_CASES)
def test_split_precision(L, name, B, h, c3, c1, cout, ups, sc):
    """Split-precision validation mode (operand_dtype fp16x3): every operand a hi / lo fp16 pair, every weight packed as
    W_hi | W_hi | W_lo, against fp64 on the fp32 operands."""
    g = torch.Generator(device="cuda").manual_seed(500 * h + c3 + c1 + ups)
    x3 = torch.randn(B, h, h, c3, device="cuda", generator=g)
    x1 = torch.randn(B, h, h, c1, device="cuda", generator=g) * 2 if c1 else None
    w3 = _weights(g, cout, c3)
    w1 = _weights(g, cout, c1, 1) if c1 else None
    bias = torch.randn(cout, device="cuda", generator=g) * 0.5
    a3, a3_lo = _split(x3)
    a1, a1_lo = _split(x1) if c1 else (None, None)
    out, stats = _conv_ex(L, a3=a3, a3_lo=a3_lo, w3=w3, bias=bias, c3=c3, cout=cout, batch=B, h=h, w=h, f16=1, a1=a1, a1_lo=a1_lo,
                          w1=w1, c1=c1, ups=ups, sc=sc)
    src = _nchw(x3.double())
    if ups:
        src = F.interpolate(src, scale_factor=2, mode="nearest")
    ref = F.conv2d(src, w3.double(), bias.double(), padding=1)
    if c1:
        ref = ref + F.conv2d(_nchw(x1.double()), w1.double())
    ref = _nhwc(ref)
    tag = f"split {name} {h} B{B} c3 {c3} c1 {c1} cout {cout} sc{sc}"
    rel, mx = _rel(out, ref), (out.double() - ref).abs().max().item()
    print(f"PARITY {tag} rel {rel:.3e} maxabs {mx:.3e}")
    assert rel <= SPLIT_REL, (tag, rel)
    if sc:
        _check_stats(L, stats, ref, B, sc, tag, parity_low=(h, h) if ups else None)


# ---------------------------------------------------------------------------------------------------- saturation
SAT_CASES = [
    # name, B, h, c, ups, resid_mode
    ("plain", 2, 16, 128, 0, 0),       # variant 6-8
    ("ups", 3, 8, 128, 1, 0),          # variants 12-14 and the generic scatter of the ragged tile
    ("resid_rep", 4, 28, 64, 0, 2),    # generic
    ("resid_up", 3, 14, 64, 0, 1),     # generic
]


@pytest.mark.parametrize("f16", [1, 0])
@pytest.mark.parametrize("name,B,h,c,ups,mode", SAT_CASES)
def test_fp16_saturation(L, name, B, h, c, ups, mode, f16):
    """A 16-bit fp16 output driven past 65504 by the bias is clamped to +-65504, never inf, and counted; bf16 counts nothing."""
    g = torch.Generator(device="cuda").manual_seed(600 + h)
    x = _act(g, B, h, h, c, f16)
    w = _weights(g, c, c)
    bias = torch.full((c,), 1.0e5, device="cuda")
    bias[1::2] = -1.0e5
    res = None
    if mode == 1:
        res = torch.randn(B, h // 2, h // 2, c, device="cuda", generator=g)
    elif mode == 2:
        res = torch.randn(B // 2, h, h, c, device="cuda", generator=g)
    sat = torch.zeros(1, device="cuda", dtype=torch.int64)
    out, _ = _conv_ex(L, a3=x, w3=w, bias=bias, c3=c, cout=c, batch=B, h=h, w=h, f16=f16, ups=ups, residual=res, resid_mode=mode,
                      out16=True, sat=sat)
    n = sat.item()
    assert torch.isfinite(out.float()).all(), name
    if f16:
        assert torch.equal(out[..., 0::2].float().unique(), torch.tensor([65504.0], device="cuda")), name
        assert torch.equal(out[..., 1::2].float().unique(), torch.tensor([-65504.0], device="cuda")), name
        assert n > 0, name
    else:
        assert n == 0, (name, n)
        assert (out[..., 0::2].float() - 1e5).abs().max().item() <= 1e5 * U16[0] + 64, name


# ---------------------------------------------------------------------------------------------------- in_conv / out_conv
IN_CASES = [
    # B, C, H, hid
    (3, 3, 32, 256),     # CIFAR
    (3, 1, 28, 64),      # MNIST-style
    (2, 3, 64, 192),     # CelebA
    (3, 6, 16, 128),
    (2, 6, 32, 64),
]


@pytest.mark.parametrize("f16", [1, 0])
@pytest.mark.parametrize("rep", [1, 2])
@pytest.mark.parametrize("B,Cin,H,hid", IN_CASES)
def test_in_conv(L, B, Cin, H, hid, rep, f16):
    """in_conv: im2col into 64 patch columns (output image i reads input image i / rep) and the pointwise GEMM, with the
    statistics the first GroupNorm reads."""
    g = torch.Generator(device="cuda").manual_seed(700 + H + Cin + hid)
    x = torch.randn(B, Cin, H, H, device="cuda", generator=g)
    w = _weights(g, hid, Cin)
    bias = torch.randn(hid, device="cuda", generator=g) * 0.5
    sc = 4 if (hid // 32) % 4 == 0 else 2
    n = B * rep
    slabs = L.vdt_stat_slabs_per_image(H, H)
    out = torch.full((n, H, H, hid), float("nan"), device="cuda")
    stats = torch.full((n * slabs + 4, hid // sc, 2), float("nan"), device="cuda")
    _check(L, L.vdt_op_in_conv(C.c_void_p(x.data_ptr()), B, rep, Cin, H, H, C.c_void_p(w.data_ptr()), C.c_void_p(bias.data_ptr()), hid,
                               C.c_void_p(out.data_ptr()), C.c_void_p(stats.data_ptr()), sc, f16, None))
    torch.cuda.synchronize()
    ref = _nhwc(F.conv2d(x.to(DT[f16]).double(), w.to(DT[f16]).double(), bias.double(), padding=1)).repeat_interleave(rep, dim=0)
    tag = f"in_conv {H} B{B} C{Cin} rep{rep} hid{hid} {FMT[f16]}"
    _check_out(out, ref, f16, tag)
    _check_stats(L, stats, ref, n, sc, tag)
    _check_groupnorm(L, out, stats, ref, n, sc, f16, tag)


OUT_CASES = [
    # B, H, c0, Cout
    (3, 32, 256, 3),     # CIFAR
    (3, 28, 64, 1),      # MNIST-style
    (2, 64, 192, 6),     # CelebA "both" output
    (3, 16, 128, 6),
    (2, 16, 64, 3),
]


@pytest.mark.parametrize("f16", [1, 0])
@pytest.mark.parametrize("B,H,c0,Cout", OUT_CASES)
def test_out_conv(L, B, H, c0, Cout, f16):
    """out_conv: the pointwise GEMM over tap-major weight rows (padded to a multiple of 32) and the tap sum into NCHW,
    including the zero padding at every border."""
    g = torch.Generator(device="cuda").manual_seed(800 + H + c0 + Cout)
    a = _act(g, B, H, H, c0, f16)
    w = _weights(g, Cout, c0)
    bias = torch.randn(Cout, device="cuda", generator=g)
    out = torch.full((B, Cout, H, H), float("nan"), device="cuda")
    _check(L, L.vdt_op_out_conv(C.c_void_p(a.data_ptr()), B, H, H, c0, C.c_void_p(w.data_ptr()), Cout, C.c_void_p(bias.data_ptr()),
                                C.c_void_p(out.data_ptr()), f16, None))
    torch.cuda.synchronize()
    ref = F.conv2d(_nchw(a.double()), w.to(DT[f16]).double(), bias.double(), padding=1)
    tag = f"out_conv {H} B{B} c0 {c0} Cout {Cout} {FMT[f16]}"
    _check_out(out, ref, f16, tag)
