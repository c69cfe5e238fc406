"""The ctypes bindings are parsed from include/tensorgame.h: every declared function is bound with the header's types,
and a type the parser does not know is refused instead of guessed."""
import ctypes as C

import pytest

from mat_mul_b200 import _lib

P = C.c_void_p


def test_every_declared_function_is_bound():
    L = _lib.lib()
    names = _lib.exported_symbols()
    assert names == sorted(_lib._SIGNATURES) and len(names) >= 69
    for name in names:
        res, args = _lib._SIGNATURES[name]
        fn = getattr(L, name)
        assert fn.restype is res and list(fn.argtypes) == args, name


def test_pinned_signatures():
    sig = _lib._SIGNATURES
    ints = [C.c_int] * 6
    assert sig["tg_demo_gen_box"] == (C.c_int, [C.c_uint64, C.c_uint64, C.c_int64, *ints, P, P, C.c_int, C.c_int, P,
                                                C.c_int64, P, P, P])
    assert sig["tg_demo_from_ustream_workspace"] == (C.c_int64, [C.c_int64, C.c_int])
    assert sig["tg_error_string"] == (C.c_char_p, [C.c_int])
    assert sig["tg_host_ctx_create"] == (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int64])
    assert sig["tg_layout"] == (C.c_int, [C.c_int] + [C.POINTER(C.c_int)] * 3)
    assert sig["tg_version"] == (C.c_int, [])
    assert sig["tg_sample_unimodular"][1][4] is C.c_double and sig["tg_mt19937_fill_f64"][1][0] is C.c_uint32


def test_parser_reads_comments_and_refuses_unknown_types():
    text = "/* int tg_hidden(int x); */\nint tg_ok(const uint8_t *tape, /* the batch */ int64_t B,\n  void *stream);\n"
    assert _lib._parse_prototypes(text) == {"tg_ok": (C.c_int, [P, C.c_int64, P])}
    for bad in ("int tg_bad(float x, void *stream);", "size_t tg_bad(int x);", "long tg_bad(void);"):
        with pytest.raises(_lib.TensorGameError, match="no ctypes type"):
            _lib._parse_prototypes(bad)
