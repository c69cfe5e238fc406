"""The inverse triples without a GPU: tests/basis_inverse_ref.py pinned to numpy.linalg.inv and an exact M X = I on sampled
triples, its predicate at the edges, the GF(2) wrapper, and the argument rules of tg_invert_bases and tg_invert_bases_gf2
in a child process that sees no CUDA device."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from mat_mul_b200 import _lib
from oracle import tg_oracle as orc
from tests import basis_inverse_ref as ref
from tests import gf2_basis_ref
from tests.test_cabi_args import BAD_SIZES, E_ARG, OK, ROOT, ptr

INT_SIZES = (4, 9, 16)
GF2_SIZES = (4, 9, 16, 25)


@pytest.mark.parametrize("S", INT_SIZES)
@pytest.mark.parametrize("p", (0.1, 0.3))
def test_fraction_reference_matches_numpy_on_sampled_triples(S, p):
    n = 12 if S == 16 else 30
    M = orc.sample_unimodular(3, (1 << 32) - 5, n, S, p).astype(np.int64).reshape(-1, S, S)
    for m in M:
        X = ref.inverse_int8(m)
        Y = np.rint(np.linalg.inv(m.astype(np.float64))).astype(np.int64)
        assert np.array_equal(m @ Y, np.eye(S, dtype=np.int64))  # unimodular: the rounded inverse is exact
        if np.abs(Y).max() <= 127 and Y.min() >= -128:
            assert np.array_equal(X, Y)
        else:
            assert X is None


@pytest.mark.parametrize("S", INT_SIZES)
def test_batch_reference_is_the_fraction_reference(S):
    """inverses_int8 (float screen + exact certificate, fractions otherwise) against inverse_int8 matrix by matrix"""
    rng = np.random.default_rng(S)
    M = orc.sample_unimodular(5, 0, 6, S, 1.0).astype(np.int64)  # dense triangles: mostly too large for int8
    edges = np.stack([m for _, m, _ in ref.integer_edges(S, rng)])
    E = np.stack([edges, np.roll(edges, 1, 0), np.roll(edges, 2, 0)], 1)
    R = rng.integers(-2, 3, size=(4, 3, S, S))  # random integer matrices: mostly det not +-1
    for mats in (M, E, R):
        inv, flags = ref.inverses_int8(mats)
        for n in range(mats.shape[0]):
            want = [ref.inverse_int8(mats[n, f]) for f in range(3)]
            assert flags[n] == (ref.FLAG_SINGULAR if any(w is None for w in want) else 0)
            for f in range(3):
                assert np.array_equal(inv[n, f], np.zeros((S, S), np.int64) if want[f] is None else want[f])


@pytest.mark.parametrize("S", INT_SIZES)
def test_integer_edges(S):
    for label, m, has in ref.integer_edges(S, np.random.default_rng(10 + S)):
        X = ref.inverse_int8(m)
        assert (X is not None) == has, label
        if has:
            assert np.array_equal(m @ X, np.eye(S, dtype=np.int64)), label
    assert ref.inverse_int8(ref._chain(S, -127, -1)).max() == 127
    assert ref.inverse_int8(ref._chain(S, -16, 8)).min() == -128


@pytest.mark.parametrize("S", (9, 16))
def test_an_edge_needs_the_exact_product_check(S):
    """The lifted inverse of mod_p_impostor modulo 32749 passes the int8 range test, so a kernel without the M X = I check
    would return it as the inverse"""
    m = ref.mod_p_impostor(S)
    assert ref.inverse_int8(m) is None and round(np.linalg.det(m)) == 1
    r, invertible = ref._inverses_mod_p(m[None], 32749)
    X = np.where(r[0] > 32749 // 2, r[0] - 32749, r[0])
    assert invertible[0] and X.min() >= -128 and X.max() <= 127
    assert not np.array_equal(m @ X, np.eye(S, dtype=np.int64))
    assert any(label.startswith("inverse mod 32749") for label, _, _ in ref.integer_edges(S, np.random.default_rng(0)))


@pytest.mark.parametrize("S", GF2_SIZES)
def test_gf2_reference(S):
    rng = np.random.default_rng(20 + S)
    M = rng.integers(0, 2, size=(20, S, S))
    singular = 0
    for m in M:
        X = ref.inverse_gf2_or_none(m)
        if X is None:
            singular += 1
            with pytest.raises(AssertionError):
                gf2_basis_ref.inverse_gf2(m)
        else:
            assert np.array_equal((m @ X) & 1, np.eye(S, dtype=np.int64))
    assert 0 < singular < 20  # about 71 % of random 0/1 matrices are singular over GF(2)
    bits = gf2_basis_ref.mats_to_bits(M[:18].reshape(6, 3, S, S))
    inv, flags = ref.inverses_gf2(bits, S)
    for n in range(6):
        want = [ref.inverse_gf2_or_none(M[3 * n + f]) for f in range(3)]
        assert flags[n] == (ref.FLAG_SINGULAR if any(w is None for w in want) else 0)
        for f in range(3):
            assert np.array_equal(gf2_basis_ref.bits_to_mats(inv[n, f], S), 0 * M[0] if want[f] is None else want[f])


# ---------------------------------------------------------------- argument rules
ARGS = ("mats", "inv", "flags", "N", "S", "stream")


def _rows(S: int):
    """(label, entry point, arguments, expected code); each row breaks one argument and keeps the others valid."""
    n = None
    valid = dict(N=4, S=S, stream=n)
    out = []

    def add(fn, sizes, label, expect, **kw):
        a = {**valid, **kw}
        out.append((f"{fn} S={S} {label}", fn, tuple(a[k] if k in a else ptr() for k in ARGS), expect if S in sizes else E_ARG))

    for fn, sizes, align in (("tg_invert_bases", INT_SIZES, 1), ("tg_invert_bases_gf2", GF2_SIZES, 4)):
        if S not in sizes:
            add(fn, sizes, "otherwise valid", E_ARG)
        add(fn, sizes, "empty batch", OK, N=0, mats=n, inv=n, flags=n)
        add(fn, sizes, "N -1", E_ARG, N=-1)
        add(fn, sizes, "empty batch, N -1", E_ARG, N=-1, mats=n)
        add(fn, sizes, "all null", E_ARG, mats=n, inv=n, flags=n)
        for k in ("mats", "inv", "flags"):
            add(fn, sizes, f"{k} null", E_ARG, **{k: n})
        for k in ("mats", "inv"):
            for o in (1, 2, 3):
                if o % align:
                    add(fn, sizes, f"{k} at +{o}", E_ARG, **{k: ptr(o)})
    return out


def table():
    return [r for S in GF2_SIZES + BAD_SIZES for r in _rows(S)]


def _run_table() -> None:
    """Child process: every row's return code, as JSON on stdout."""
    assert os.environ.get("CUDA_VISIBLE_DEVICES") == "", "the table runs only where no device is visible"
    L = _lib.lib()
    print(json.dumps({label: getattr(L, fn)(*args) for label, fn, args, _ in table()}))


def test_argument_rules_of_the_basis_inversions():
    rows = table()
    assert len({r[0] for r in rows}) == len(rows)
    assert any(r[0] == "tg_invert_bases S=25 otherwise valid" and r[3] == E_ARG for r in rows)
    res = subprocess.run([sys.executable, "-c", "from tests.test_basis_inverse_ref import _run_table; _run_table()"], cwd=ROOT,
                         env={**os.environ, "CUDA_VISIBLE_DEVICES": ""}, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr
    got = json.loads(res.stdout.strip().splitlines()[-1])
    wrong = [f"{label}: {got[label]}, want {want}" for label, _, _, want in rows if got[label] != want]
    assert not wrong, f"{len(wrong)} of {len(rows)} calls:\n" + "\n".join(wrong)
