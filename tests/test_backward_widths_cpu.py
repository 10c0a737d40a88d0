"""CPU: the width checks of the two backward entry points that take the UNet's channel counts -- GroupNorm backward (C % 64 == 0,
C <= 2048) and wgrad (cout % 64 == 0) -- refuse out-of-range widths through vdt_last_error before any device call."""
import ctypes as C

from v_diffusion_b200 import _lib

DUMMY = C.c_void_p(0x1000)          # never dereferenced: the width check fires first


def test_groupnorm_backward_refuses_widths_off_the_64_grid():
    L = _lib.lib()
    for c in (96, 32, 2112):
        rc = L.vdt_op_groupnorm_backward(DUMMY, DUMMY, c, 2, 8, 8, DUMMY, DUMMY, None, 1, C.c_float(0.0), 0, 0, DUMMY, DUMMY, DUMMY,
                                         None, None)
        assert rc != 0
        msg = L.vdt_last_error().decode()
        assert "multiple of 64 channels up to 2048" in msg and f"got {c}" in msg, msg


def test_wgrad_refuses_cout_off_the_64_grid():
    L = _lib.lib()
    rc = L.vdt_op_conv_wgrad(DUMMY, DUMMY, 2, 16, 16, 64, 96, 3, DUMMY, DUMMY, 1, None)
    assert rc != 0
    msg = L.vdt_last_error().decode()
    assert "cout % 64 == 0" in msg and "64 -> 96" in msg, msg
