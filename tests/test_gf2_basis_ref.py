"""The change of basis over GF(2) without a GPU: tests/gf2_basis_ref.py pinned to the C oracle's integer change of basis,
factor transform and unimodular sampler taken mod 2 (at 4, 9 and 16), its algebra at every size, 25 included, and the
argument rules of the three entry points."""
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest

from mat_mul_b200 import _lib
from oracle import tg_oracle as orc
from tests import gf2_basis_ref as ref
from tests import gf2_ref
from tests.test_cabi_args import BAD_SIZES, E_ARG, OK, ROOT, ptr

SIZES = (4, 9, 16, 25)
ORACLE_SIZES = (4, 9, 16)  # orc_sample_unimodular and the integer change of basis stop at 16
PROBS = (0.0, 1 / 128, 0.3, 1.0)
FIRST = (1 << 32) - 2  # games 0 and 1 have d_hi = 0, games 2.. have d_hi = 1: the key changes within the batch
SEED = 0x0123456789ABCDEF


def _int_mats(S, n, rng):
    """integer triples with negative entries"""
    return rng.integers(-3, 4, size=(n, 3, S, S))


@pytest.mark.parametrize("S", ORACLE_SIZES)
def test_transform_is_the_oracle_change_of_basis_mod_2(S):
    rng = np.random.default_rng(S)
    T = rng.integers(-9, 10, size=(3, S, S, S))
    M = _int_mats(S, 3, rng)
    want = np.stack([orc.change_of_basis(T[n], M[n, 0], M[n, 1], M[n, 2]) & 1 for n in range(3)])
    assert np.array_equal(ref.transform(T, M), want)
    assert np.array_equal(ref.transform(T, M[:1]), np.stack([orc.change_of_basis(t, *M[0]) & 1 for t in T]))  # shared


@pytest.mark.parametrize("S", ORACLE_SIZES)
def test_factor_transform_is_the_oracle_mod_2(S):
    rng = np.random.default_rng(10 + S)
    N, R = 3, 5
    for shift_in, shift_out in ((1, 1), (4, 2), (3, 4)):
        val = rng.integers(-shift_in, 5 - shift_in, size=(N, R, 3 * S))  # coefficients of both signs, tokens in [0, 4]
        M = _int_mats(S, N, rng)
        got = ref.factors(val + shift_in, M, shift_in, shift_out)
        for n in range(N):
            want = orc.change_of_basis_factors(val[n].reshape(R, 3, S), *M[n]) & 1
            assert np.array_equal(got[n] - shift_out, want.reshape(R, 3 * S)), (shift_in, shift_out, n)


@pytest.mark.parametrize("S", ORACLE_SIZES)
@pytest.mark.parametrize("p", PROBS)
def test_sampler_is_the_unimodular_sampler_mod_2(S, p):
    want = orc.sample_unimodular(SEED, FIRST, 5, S, p) & 1
    assert np.array_equal(ref.sample_invertible(SEED, FIRST, 5, S, p), want)


@pytest.mark.parametrize("S", SIZES)
def test_sampled_matrices_are_invertible(S):
    for p in PROBS:
        M = ref.sample_invertible(SEED, FIRST, 4, S, p)
        assert all(gf2_ref.rank_gf2(m) == S for m in M.reshape(-1, S, S)), p
        if p == 0:
            assert np.array_equal(M, np.broadcast_to(np.eye(S, dtype=np.int64), M.shape))
        for m in M.reshape(-1, S, S):
            assert np.array_equal((ref.inverse_gf2(m) @ m) & 1, np.eye(S, dtype=np.int64))
    dense = ref.sample_invertible(7, 0, 6, S, 1.0)  # every draw non-zero: L and U are full triangles
    assert not np.array_equal(dense, np.broadcast_to(np.eye(S, dtype=np.int64), dense.shape))


@pytest.mark.parametrize("S", SIZES)
def test_bit_matrices_round_trip_and_ignore_high_bits(S):
    rng = np.random.default_rng(20 + S)
    M = rng.integers(-5, 6, size=(4, 3, S, S))
    bits = ref.mats_to_bits(M)
    assert bits.shape == (4, 3, S) and np.array_equal(ref.bits_to_mats(bits, S), M & 1)
    assert not (bits.view(np.uint32) >> S).any()
    junk = (bits.view(np.uint32) | (rng.integers(0, 1 << 32, size=bits.shape, dtype=np.uint64).astype(np.uint32) & ~np.uint32((1 << S) - 1)))
    assert np.array_equal(ref.bits_to_mats(junk.view(np.int32), S), M & 1)


@pytest.mark.parametrize("S", SIZES)
def test_bases_then_their_inverses_return_the_tensor(S):
    rng = np.random.default_rng(30 + S)
    T = rng.integers(0, 2, size=(3, S, S, S))
    M = ref.sample_invertible(5, 0, 3, S, 0.3)
    Minv = np.stack([[ref.inverse_gf2(M[n, f]) for f in range(3)] for n in range(3)])
    Tp = ref.transform(T, M)
    assert not np.array_equal(Tp, T)
    assert np.array_equal(ref.transform(Tp, Minv), T)


@pytest.mark.parametrize("S", SIZES)
def test_transformed_tape_sums_to_the_transformed_tensor(S):
    rng = np.random.default_rng(40 + S)
    N, R = 3, 9
    for shift_in, shift_out in ((1, 3), (4, 4)):
        tok = rng.integers(0, 256, size=(N, R, 3 * S))
        M = ref.sample_invertible(9, 4, N, S, 0.5)
        Tp = ref.transform(ref.rank1_sum(tok, shift_in), M)
        tok2 = ref.factors(tok, M, shift_in, shift_out)
        assert tok2.min() >= shift_out and tok2.max() <= shift_out + 1
        assert np.array_equal(ref.rank1_sum(tok2, shift_out), Tp)


# ---------------------------------------------------------------- argument rules
BASIS = ("in", "mats", "per_game", "out", "N", "S", "stream")
FACTORS = ("tin", "istride", "shift_in", "mats", "per_game", "tout", "ostride", "shift_out", "N", "R", "S", "stream")
SAMPLE = ("seed", "first", "N", "S", "p", "mats", "stream")


def _rows(S: int):
    """(label, entry point, arguments, expected code); each row breaks one argument and keeps the others valid."""
    n = None
    valid = dict(N=4, S=S, per_game=1, istride=64, ostride=64, shift_in=2, shift_out=3, R=2, seed=SEED, first=FIRST, p=0.3,
                 stream=n)
    out = []

    def add(fn, names, label, expect, **kw):
        a = {**valid, **kw}
        out.append((f"{fn} S={S} {label}", fn, tuple(a[k] if k in a else ptr() for k in names), expect if S in SIZES else E_ARG))

    def common(fn, names, pointers, aligned):
        if S not in SIZES:
            add(fn, names, "otherwise valid", E_ARG)
        add(fn, names, "empty batch", OK, N=0, **{k: n for k in pointers})
        add(fn, names, "N -1", E_ARG, N=-1)
        add(fn, names, "all null", E_ARG, **{k: n for k in pointers})
        for k in pointers:
            add(fn, names, f"{k} null", E_ARG, **{k: n})
        for k, align in aligned.items():
            for o in (1, 2, 4, 8):
                if o % align:
                    add(fn, names, f"{k} at +{o}", E_ARG, **{k: ptr(o)})

    common("tg_change_of_basis_gf2", BASIS, ("in", "mats", "out"), {"in": 16, "out": 16, "mats": 4})
    add("tg_change_of_basis_gf2", BASIS, "shared triple, empty batch", OK, N=0, per_game=0)

    fn = "tg_change_of_basis_factors_gf2"
    common(fn, FACTORS, ("tin", "mats", "tout"), {"tin": 16, "tout": 16, "mats": 4})
    for k in ("shift_in", "shift_out"):
        for sh in (0, 5, 9, -1):
            add(fn, FACTORS, f"{k} {sh}", E_ARG, **{k: sh})
        add(fn, FACTORS, f"empty batch, {k} 0", E_ARG, N=0, **{k: 0})
    for r in (0, -1):
        add(fn, FACTORS, f"R {r}", E_ARG, R=r)
    add(fn, FACTORS, "empty batch, R 0", E_ARG, N=0, R=0)
    for k in ("istride", "ostride"):
        for st in (4, 8, 40):
            add(fn, FACTORS, f"{k} {st}", E_ARG, **{k: st})

    fn = "tg_sample_invertible_gf2"
    common(fn, SAMPLE, ("mats",), {"mats": 4})
    for p in (-0.01, 1.01, math.nan, math.inf, -math.inf):
        add(fn, SAMPLE, f"p {p}", E_ARG, p=p)
    add(fn, SAMPLE, "empty batch, p nan", E_ARG, N=0, p=math.nan)
    for p in (0.0, 1.0):
        add(fn, SAMPLE, f"empty batch, p {p}", OK, N=0, p=p)
    return out


def table():
    return [r for S in SIZES + BAD_SIZES for r in _rows(S)]


def _run_table() -> None:
    """Child process: every row's return code, as JSON on stdout."""
    assert os.environ.get("CUDA_VISIBLE_DEVICES") == "", "the table runs only where no device is visible"
    L = _lib.lib()
    print(json.dumps({label: getattr(L, fn)(*args) for label, fn, args, _ in table()}))


def test_argument_rules_of_the_change_of_basis_mod_2():
    rows = table()
    assert len({r[0] for r in rows}) == len(rows)
    res = subprocess.run([sys.executable, "-c", "from tests.test_gf2_basis_ref import _run_table; _run_table()"], cwd=ROOT,
                         env={**os.environ, "CUDA_VISIBLE_DEVICES": ""}, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr
    got = json.loads(res.stdout.strip().splitlines()[-1])
    wrong = [f"{label}: {got[label]}, want {want}" for label, _, _, want in rows if got[label] != want]
    assert not wrong, f"{len(wrong)} of {len(rows)} calls:\n" + "\n".join(wrong)
