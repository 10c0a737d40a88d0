"""CPU: every refusal of the conv-mode hooks (vdt_op_conv_ex, vdt_op_in_conv, vdt_op_out_conv).  They check their
arguments before any CUDA call, so the refusals come back through vdt_last_error without a device (the pointers below
are never dereferenced)."""
import ctypes as C

import pytest

from v_diffusion_b200 import _lib

P = [C.c_void_p(0x10000 * (i + 1)) for i in range(8)]      # distinct non-null stand-ins for device pointers


def _base(**kw):
    f = dict(a3=P[0], w3=P[1], bias=P[2], out_f32=P[3], batch=2, h=16, w=16, c3=64, c1=0, cout=64, ups=0, resid_mode=0,
             stat_cols=4, f16=1)
    f.update(kw)
    return _lib.ConvOp(**{k: (v.value if isinstance(v, C.c_void_p) else v) for k, v in f.items()})


CONV_EX_REFUSALS = {
    "ups_with_skip": (dict(ups=1, a1=P[4], w1=P[5], c1=64), "no 1x1 skip"),
    "ups_with_residual": (dict(ups=1, residual=P[4]), "no residual"),
    "resid_rep_with_ups": (dict(ups=1, residual=P[4], resid_mode=2), "no residual"),
    "resid_up_odd_sides": (dict(h=15, w=15, residual=P[4], resid_mode=1), "even output sides"),
    "resid_up_odd_width": (dict(h=16, w=14 + 1, residual=P[4], resid_mode=1), "even output sides"),
    "resid_rep_odd_batch": (dict(batch=3, residual=P[4], resid_mode=2), "even batch"),
    "resid_mode_without_residual": (dict(resid_mode=1), "needs a residual"),
    "resid_mode_unknown": (dict(residual=P[4], resid_mode=3), "resid_mode must be"),
    "a3_lo_without_a1_lo": (dict(a3_lo=P[4], a1=P[5], w1=P[6], c1=64), "split-precision"),
    "a1_lo_without_a3_lo": (dict(a1=P[5], a1_lo=P[4], w1=P[6], c1=64), "split-precision"),
    "a1_lo_without_a1": (dict(a1_lo=P[4]), "a1_lo without a1"),
    "a1_without_w1": (dict(a1=P[5], c1=64), "come together"),
    "w1_without_a1": (dict(w1=P[5], c1=64), "come together"),
    "c3_off_grid": (dict(c3=96), "multiples of 64"),
    "cout_off_grid": (dict(cout=32), "multiples of 64"),
    "c1_off_grid": (dict(a1=P[4], w1=P[5], c1=32), "multiples of 64"),
    "no_output": (dict(out_f32=None), "exactly one"),
    "two_outputs": (dict(out16=P[4]), "exactly one"),
    "no_weights": (dict(w3=None), "required"),
    "f16_flag": (dict(f16=2), "f16 must be"),
    "ups_flag": (dict(ups=2), "ups must be"),
    "empty": (dict(batch=0), "empty input"),
    "too_wide": (dict(h=2, w=200), "feature-map width"),
    "stats_7x7": (dict(h=7, w=7, stats=P[4]), "statistics layout"),
    "stats_4x4": (dict(h=4, w=4, stats=P[4]), "statistics layout"),
    "stats_ups_7_to_14": (dict(h=7, w=7, ups=1, stats=P[4]), "statistics layout"),
    "stats_ups_14_to_28": (dict(h=14, w=14, ups=1, stats=P[4]), "statistics layout"),     # 4 * 8 slabs != 28
    "stats_ups_4_to_8": (dict(h=4, w=4, ups=1, stats=P[4]), "statistics layout"),
    "stat_cols": (dict(stats=P[4], stat_cols=3), "stat_cols must be"),
}


@pytest.mark.parametrize("name", sorted(CONV_EX_REFUSALS))
def test_conv_ex_refusals(name):
    L = _lib.lib()
    kw, msg = CONV_EX_REFUSALS[name]
    op = _base(**kw)
    assert L.vdt_op_conv_ex(C.byref(op), None) != 0
    assert msg in L.vdt_last_error().decode(), L.vdt_last_error().decode()


def test_conv_ex_refuses_null_op():
    L = _lib.lib()
    assert L.vdt_op_conv_ex(None, None) != 0 and b"null" in L.vdt_last_error()


def _in_conv(L, x=P[0], batch=2, rep=1, c=3, h=16, w=16, hid=64, stats=None, stat_cols=4, f16=1):
    return L.vdt_op_in_conv(x, batch, rep, c, h, w, P[1], P[2], hid, P[3], stats, stat_cols, f16, None)


IN_CONV_REFUSALS = {
    "null_input": (dict(x=None), "null argument"),
    "rep_3": (dict(rep=3), "rep must be"),
    "too_many_channels": (dict(c=8), "1 to 7 input channels"),
    "no_channels": (dict(c=0), "1 to 7 input channels"),
    "hid_off_grid": (dict(hid=96), "multiples of 64"),
    "f16_flag": (dict(f16=-1), "f16 must be"),
    "empty": (dict(h=0), "empty input"),
    "stats_7x7": (dict(h=7, w=7, stats=P[4]), "statistics layout"),
    "stat_cols": (dict(stats=P[4], stat_cols=1), "stat_cols must be"),
}


@pytest.mark.parametrize("name", sorted(IN_CONV_REFUSALS))
def test_in_conv_refusals(name):
    L = _lib.lib()
    kw, msg = IN_CONV_REFUSALS[name]
    assert _in_conv(L, **kw) != 0
    assert msg in L.vdt_last_error().decode(), L.vdt_last_error().decode()


def _out_conv(L, a=P[0], batch=2, h=16, w=16, c0=64, cout=3, f16=1):
    return L.vdt_op_out_conv(a, batch, h, w, c0, P[1], cout, P[2], P[3], f16, None)


OUT_CONV_REFUSALS = {
    "null_input": (dict(a=None), "null argument"),
    "c0_off_grid": (dict(c0=96), "multiples of 64"),
    "too_many_outputs": (dict(cout=17), "1 to 16 output channels"),
    "no_outputs": (dict(cout=0), "1 to 16 output channels"),
    "f16_flag": (dict(f16=3), "f16 must be"),
    "empty": (dict(batch=0), "empty input"),
}


@pytest.mark.parametrize("name", sorted(OUT_CONV_REFUSALS))
def test_out_conv_refusals(name):
    L = _lib.lib()
    kw, msg = OUT_CONV_REFUSALS[name]
    assert _out_conv(L, **kw) != 0
    assert msg in L.vdt_last_error().decode(), L.vdt_last_error().decode()
