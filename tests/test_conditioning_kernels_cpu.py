"""CPU: every refusal of the conditioning-path hooks (vdt_op_timestep_embedding_ex, vdt_op_class_embed, vdt_op_film_rows,
vdt_op_multitag_rows, vdt_op_attention_f32) and of vdt_op_linear's shape limits, and the ctypes signatures against the
header.  The hooks check their arguments before any CUDA call, so the refusals come back through vdt_last_error without a
device (the pointers below are never dereferenced)."""
import ctypes as C
import re

import pytest

from v_diffusion_b200 import _lib

P = [C.c_void_p(0x10000 * (i + 1)) for i in range(8)]      # distinct non-null stand-ins for device pointers


def _refused(L, rc, msg):
    assert rc != 0
    assert msg in L.vdt_last_error().decode(), L.vdt_last_error().decode()


def _linear(L, x=P[0], w=P[1], b=P[2], out=P[3], rows=4, k=64, n=8):
    return L.vdt_op_linear(x, w, b, out, rows, k, n, 0, None)


LINEAR_REFUSALS = {
    "k_1537": (dict(k=1537), "exceeds the 1536 columns"),
    "k_zero": (dict(k=0), "bad linear shape"),
    "n_zero": (dict(n=0), "bad linear shape"),
    "rows_negative": (dict(rows=-1), "bad linear shape"),
    "null_x": (dict(x=None), "null argument"),
    "null_bias": (dict(b=None), "null argument"),
}


@pytest.mark.parametrize("name", sorted(LINEAR_REFUSALS))
def test_linear_refusals(name):
    L = _lib.lib()
    kw, msg = LINEAR_REFUSALS[name]
    _refused(L, _linear(L, **kw), msg)


def _temb(L, t=P[0], out=P[1], rows=4, dim=64, fp32_t=0):
    return L.vdt_op_timestep_embedding_ex(t, out, rows, dim, fp32_t, None)


TEMB_REFUSALS = {
    "null_t": (dict(t=None), "null argument"),
    "null_out": (dict(out=None), "null argument"),
    "rows_negative": (dict(rows=-1), "bad embedding shape"),
    "dim_3": (dict(dim=3), "bad embedding shape"),        # dim / 2 - 1 = 0: the frequency formula divides by it
    "fp32_t_flag": (dict(fp32_t=2), "fp32_t must be"),
    "too_many_elements": (dict(rows=1 << 24, dim=256), "exceeds 2^31 - 1"),
}


@pytest.mark.parametrize("name", sorted(TEMB_REFUSALS))
def test_timestep_embedding_ex_refusals(name):
    L = _lib.lib()
    kw, msg = TEMB_REFUSALS[name]
    _refused(L, _temb(L, **kw), msg)


def test_timestep_embedding_shares_the_shape_checks():
    L = _lib.lib()
    _refused(L, L.vdt_op_timestep_embedding(P[0], P[1], 1 << 24, 256, None), "exceeds 2^31 - 1")
    _refused(L, L.vdt_op_timestep_embedding(P[0], P[1], 4, 2, None), "bad embedding shape")


def _cls(L, e=P[0], y=P[1], ym=None, w=P[2], b=P[3], ncls=10, out=P[4], rows=4, E=64):
    return L.vdt_op_class_embed(e, y, ym, w, b, ncls, out, rows, E, None)


CLS_REFUSALS = {
    "both_label_forms": (dict(ym=P[5]), "exactly one"),
    "no_label": (dict(y=None), "exactly one"),
    "null_e": (dict(e=None), "null argument"),
    "null_w": (dict(w=None), "null argument"),
    "null_b": (dict(b=None), "null argument"),
    "null_out": (dict(out=None), "null argument"),
    "no_classes": (dict(ncls=0), "bad class embedding shape"),
    "rows_negative": (dict(rows=-1), "bad class embedding shape"),
    "E_zero": (dict(E=0), "bad class embedding shape"),
    "too_many_elements": (dict(rows=1 << 22, E=1024), "exceeds 2^31 - 1"),
}


@pytest.mark.parametrize("name", sorted(CLS_REFUSALS))
def test_class_embed_refusals(name):
    L = _lib.lib()
    kw, msg = CLS_REFUSALS[name]
    _refused(L, _cls(L, **kw), msg)


FILM_ROWS_REFUSALS = {
    "null_out": (dict(out=None), "null argument"),
    "rows_negative": (dict(rows=-1), "bad FiLM row shape"),
    "ncls_negative": (dict(ncls=-1), "bad FiLM row shape"),
    "rep_3": (dict(rep=3), "rep must be"),
    "rep_0": (dict(rep=0), "rep must be"),
}


@pytest.mark.parametrize("name", sorted(FILM_ROWS_REFUSALS))
def test_film_rows_refusals(name):
    L = _lib.lib()
    kw, msg = FILM_ROWS_REFUSALS[name]
    a = dict(label=P[0], rows=4, rep=2, ncls=10, out=P[1])
    a.update(kw)
    _refused(L, L.vdt_op_film_rows(a["label"], a["rows"], a["rep"], a["ncls"], a["out"], None), msg)


MULTITAG_ROWS_REFUSALS = {
    "null_label": (dict(label=None), "null argument"),
    "null_out": (dict(out=None), "null argument"),
    "rows_negative": (dict(rows=-1), "bad multitag row shape"),
    "no_classes": (dict(ncls=0), "bad multitag row shape"),
    "rep_3": (dict(rep=3), "rep must be"),
    "too_many_elements": (dict(rows=1 << 26, ncls=40), "exceed 2^31 - 1"),
}


@pytest.mark.parametrize("name", sorted(MULTITAG_ROWS_REFUSALS))
def test_multitag_rows_refusals(name):
    L = _lib.lib()
    kw, msg = MULTITAG_ROWS_REFUSALS[name]
    a = dict(label=P[0], rows=4, rep=2, ncls=40, out=P[1])
    a.update(kw)
    _refused(L, L.vdt_op_multitag_rows(a["label"], a["rows"], a["rep"], a["ncls"], a["out"], None), msg)


def test_empty_row_sets_are_no_ops():
    L = _lib.lib()
    assert L.vdt_op_film_rows(None, 0, 1, 0, P[1], None) == 0
    assert L.vdt_op_multitag_rows(P[0], 0, 2, 40, P[1], None) == 0


ATT_REFUSALS = {
    "null_qkv": (dict(qkv=None), "null argument"),
    "null_lo": (dict(lo=None), "null argument"),
    "no_batch": (dict(batch=0), "empty input"),
    "no_tokens": (dict(n=0), "empty input"),
    "no_heads": (dict(heads=0), "empty input"),
    "d_96": (dict(d=96), "head dims 64, 128, 192 or 256"),
    "d_32": (dict(d=32), "head dims 64, 128, 192 or 256"),
    "f16_flag": (dict(f16=2), "f16 must be"),
}


@pytest.mark.parametrize("name", sorted(ATT_REFUSALS))
def test_attention_f32_refusals(name):
    L = _lib.lib()
    kw, msg = ATT_REFUSALS[name]
    a = dict(qkv=P[0], hi=P[1], lo=P[2], batch=2, n=16, heads=1, d=64, f16=1)
    a.update(kw)
    _refused(L, L.vdt_op_attention_f32(a["qkv"], a["hi"], a["lo"], a["batch"], a["n"], a["heads"], a["d"], a["f16"], None), msg)


def _declarations():
    """{name: parameter count} of every function include/vdt_b200.h declares."""
    hdr = re.sub(r"/\*.*?\*/", "", open(_lib.INCLUDE).read(), flags=re.S)
    out = {}
    for m in re.finditer(r"\b(vdt_[a-z0-9_]+)\s*\(([^()]*)\)\s*;", hdr):
        params = m.group(2).strip()
        out[m.group(1)] = 0 if params in ("", "void") else params.count(",") + 1
    return out


def test_ctypes_argtypes_have_the_headers_arity():
    """Every entry point that takes arguments has ctypes argtypes of the header's length: a missing or extra slot would
    pass garbage (or drop the stream) without any error at the call."""
    L = _lib.lib()
    decl = _declarations()
    assert set(decl) == set(_lib.EXPORTS), set(decl) ^ set(_lib.EXPORTS)
    for name, n in sorted(decl.items()):
        argtypes = getattr(L, name).argtypes
        if n == 0:
            assert not argtypes, name
            continue
        assert argtypes is not None, f"{name}: no argtypes"
        assert len(argtypes) == n, f"{name}: {len(argtypes)} argtypes, the header declares {n} parameters"
