"""Synthetic demonstrations modulo 2 without a GPU: tests/gf2_demo_ref.py pinned to the C oracle's integer contracts where
they coincide (alphabets whose only even value is 0), the library's host-side mod-2 tables against it, the distribution the
tables encode, and the argument rules of tg_demo_gen_gf2."""
import ctypes as C
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest

from mat_mul_b200 import _lib
from oracle import tg_oracle as orc
from tests import gf2_demo_ref as ref
from tests import oracle_any_s as oas
from tests.test_cabi_args import BAD_SIZES, E_ARG, OK, ROOT, ptr

V3, P3 = (-1, 0, 1), (0.15, 0.7, 0.15)
V5, P5 = (-2, -1, 0, 1, 2), (0.05, 0.10, 0.70, 0.10, 0.05)
# alphabets whose only even value is 0: the mod-2 contracts are the integer ones
ZERO_ONLY_EVEN = [(V3, P3), ((-1, 0, 1), (0.1, 0.8, 0.1)), ((0, 1), (0.6, 0.4)), ((-3, -1, 0, 1, 3), (0.1, 0.1, 0.5, 0.2, 0.1))]
TABLE_CASES = [(V3, P3), (V5, P5), ((0, 1), (0.6, 0.4)), ((-2, -1, 1, 2), (0.3, 0.2, 0.2, 0.3)), ((0, 2, 1), (0.5, 0.3, 0.2))]
FIRST = (1 << 32) - 5  # d_hi changes inside the batch
E_CUDA = -2


def lib_tables(values, probs, S):
    out = np.zeros((8, 128), dtype=np.uint16)
    v, p = np.array(values, dtype=np.int8), np.array(probs, dtype=np.float64)
    rc = _lib.lib().tg_demo_alias_tables_gf2(v.ctypes.data, p.ctypes.data, len(v), S, out.ctypes.data)
    return rc, out


@pytest.mark.parametrize("S", (4, 9, 16))
@pytest.mark.parametrize("case", range(len(ZERO_ONLY_EVEN)))
def test_restatement_is_the_integer_contract_where_0_is_the_only_even_value(S, case):
    values, probs = ZERO_ONLY_EVEN[case]
    assert ref.alias_applies(values, probs, S) == orc.alias_applies(values, probs, S)
    assert np.array_equal(ref.alias_tables(values, probs, S), orc.alias_tables(values, probs, S))
    tok, tgt, ex = ref.demos(11 + S, FIRST, 7, values, probs, 5, S, 3)
    wt, wg, wex = orc.demos_philox(11 + S, FIRST, 7, values, probs, 5, S, 3)
    assert np.array_equal(tok, wt) and np.array_equal(tgt, wg & 1) and wex == 0 and not ex.any()


@pytest.mark.parametrize("S", (4, 9, 16))
def test_restatement_of_v1_is_the_integer_contract_with_exhausted_terms(S):
    values, probs = (-1, 0, 1), (0.0004, 0.9992, 0.0004)  # P(0) > 0.999: v1, and short max_tries exhaust terms
    assert not ref.alias_applies(values, probs, S)
    tok, tgt, ex = ref.demos(5, FIRST, 40, values, probs, 3, S, 1, max_tries=2)
    wt, wg, wex = orc.demos_philox(5, FIRST, 40, values, probs, 3, S, 1, max_tries=2)
    assert np.array_equal(tok, wt) and np.array_equal(tgt, wg & 1)
    assert wex > 0 and ex.sum() > 0 and ex.sum() <= wex


def test_restatement_at_25_is_contract_v1():
    for values, probs in ((V3, P3), ((-3, -1, 0, 1, 3), (0.1, 0.1, 0.5, 0.2, 0.1))):
        tok, tgt, ex = ref.demos(3, FIRST, 4, values, probs, 6, 25, 3)
        wt, wg, wex = oas.demos_philox_v1(3, FIRST, 4, values, probs, 6, 25, 3)
        assert np.array_equal(tok, wt) and np.array_equal(tgt, wg & 1) and wex == 0


def test_restatement_conditions_factors_on_an_odd_entry():
    """V5 draws 2 and -2: every factor of every term still has an odd entry, under v2 and under v1 (a sixth value; a
    forced term is odd too)."""
    for values, probs, S in ((V5, P5, 4), (V5, P5, 9), ((-4, -2, 0, 1, 2, 4), (0.1, 0.2, 0.3, 0.1, 0.2, 0.1), 4)):
        tok, _, ex = ref.demos(1, 0, 300, values, probs, 4, S, 4)
        f = tok.reshape(300, 4, 3, S) - 4
        assert (f % 2 == 1).any(3).all() and ex.any() == (len(values) == 6)


@pytest.mark.parametrize("S", (4, 9, 16))
def test_library_tables_are_the_restatement(S):
    for values, probs in TABLE_CASES:
        rc, got = lib_tables(values, probs, S)
        assert rc == OK and np.array_equal(got, ref.alias_tables(values, probs, S)), (values, S)


def test_library_tables_refuse_where_v2_mod_2_does_not_apply():
    for values, probs, S in ((V3, P3, 25), (V5, P5, 25), ((-3, -2, -1, 1, 2, 3), (1,) * 6, 4),
                             ((-1, 0, 2, 1), (0.0004, 0.9, 0.0996, 0.0004), 9), ((-2, 0, 2), (0.2, 0.6, 0.2), 4), ((0,), (1.0,), 16)):
        assert not ref.alias_applies(values, probs, S)
        assert lib_tables(values, probs, S)[0] == E_ARG, (values, S)


def _table_dist(t):
    d = np.zeros(128)
    for o in range(128):
        thr, al = int(t[o]) & 511, int(t[o]) >> 9
        q = 1.0 if (thr == 511 and al == o) else thr / 512.0
        d[o] += q / 128
        d[al] += (1 - q) / 128
    return d


@pytest.mark.parametrize("S", (4, 9, 16))
def test_tables_encode_the_mod_2_conditional_distribution(S):
    """Group g's tilted table is P(group | every earlier group of the factor even) of a factor conditioned on an odd entry:
    P(x) (1 - P(every later entry even)) for an all-even x, P(x) otherwise, normalised.  A 9-bit threshold rounds a bucket's
    share by at most 2^-17; the mod-2 tilt moves mass onto the odd outcomes, which are then the alias of many buckets (V5
    at 4: 2^-12.9 off), hence 2^-12 where the integer tables hold 2^-13."""
    for values, probs in TABLE_CASES:
        n, pn = len(values), np.array(probs, dtype=np.float64) / np.sum(probs)
        pe = pn[np.array(values) % 2 == 0].sum()
        tab = ref.alias_tables(values, probs, S)
        ng = (S + 2) // 3
        last = S - 3 * (ng - 1)
        p3 = np.array([pn[o % n] * pn[(o // n) % n] * pn[o // (n * n)] for o in range(n ** 3)])
        ev3 = np.array([all(values[i] % 2 == 0 for i in (o % n, (o // n) % n, o // (n * n))) for o in range(n ** 3)])
        ev1 = np.array([v % 2 == 0 for v in values])
        assert np.abs(_table_dist(tab[0])[: n ** 3] - p3).max() < 2.0 ** -13
        assert np.abs(_table_dist(tab[1])[:n] - pn).max() < 2.0 ** -13
        for g in range(ng):
            size = 3 if g < ng - 1 else last
            base, ev = (p3, ev3) if size == 3 else (pn, ev1)
            want = base * np.where(ev, 1 - pe ** (S - 3 * g - size), 1.0)
            got = _table_dist(tab[2 + g])[: len(base)]
            assert np.abs(got - want / want.sum()).max() < 2.0 ** -12, (values, S, g)
        # the last group's tilted table never yields an all-even outcome: a factor cannot end without an odd entry
        ev_last = ev3 if last == 3 else ev1
        assert _table_dist(tab[2 + ng - 1])[: len(ev_last)][ev_last].sum() == 0.0


# ---------------------------------------------------------------- argument rules
SIZES = (4, 9, 16, 25)
_KEEP = []  # host arrays the child's calls point at


def _host(values, probs):
    v, p = np.array(values, dtype=np.int8), np.array(probs, dtype=np.float64)
    _KEEP.extend((v, p))
    return C.c_void_p(v.ctypes.data), C.c_void_p(p.ctypes.data), len(v)


def _rows(S):
    out = []
    good_v, good_p, good_n = _host(V3, P3)

    def add(label, want, N=8, R=7, shift=1, values=None, n=None, max_tries=64, tape=0, stride=8 * 32 * 16, bits=0,
            flags=0, null=()):
        vp = (good_v, good_p, good_n) if values is None else _host(*values)
        v, p, nv = vp[0], vp[1], vp[2] if n is None else n
        args = (C.c_uint64(1), C.c_uint64(0), C.c_int64(N), R, S, shift, None if "values" in null else v,
                None if "probs" in null else p, nv, max_tries, None if "tape" in null else ptr(tape), C.c_int64(stride),
                None if "bits" in null else ptr(bits), None if "flags" in null else ptr(flags), None)
        out.append((f"S {S}: {label}", args, want))

    ok = E_CUDA if S in SIZES else E_ARG  # valid arguments reach the device, which the child process does not see
    add("valid", ok)
    add("valid, flags NULL", ok, null=("flags",))
    add("valid, R 65535", ok, R=65535)
    for k, bad in (("N", -1), ("R", 0), ("R", -1), ("R", 65536), ("shift", 0), ("shift", 5), ("n", 0), ("n", 9),
                   ("max_tries", 0), ("max_tries", 65536)):
        add(f"{k} {bad}", E_ARG, **{k: bad})
        if k != "N":
            add(f"empty batch, {k} {bad}", E_ARG, N=0, **{k: bad})
    add("empty batch", OK if S in SIZES else E_ARG, N=0, null=("values", "probs", "tape", "bits"))
    add("empty batch, all-even alphabet", OK if S in SIZES else E_ARG, N=0, values=((0, 2), (0.5, 0.5)))
    for k in ("values", "probs", "tape", "bits"):
        add(f"{k} NULL", E_ARG, null=(k,))
    for k, off in (("tape", 4), ("tape", 8), ("bits", 4), ("bits", 12), ("stride", 8 * 32 * 16 + 4)):
        add(f"{k} misaligned {off}", E_ARG, **{k: off})
    add("value beyond shift", E_ARG, values=((-2, 0, 1), P3))
    add("value beyond shift 2", E_ARG, values=((-1, 0, 3), P3), shift=2)
    add("value at shift 4", ok, values=((-4, 0, 3), P3), shift=4)
    add("negative probability", E_ARG, values=(V3, (0.5, -0.1, 0.6)))
    add("NaN probability", E_ARG, values=(V3, (0.5, math.nan, 0.5)))
    add("zero probabilities", E_ARG, values=(V3, (0.0, 0.0, 0.0)))
    add("all-even alphabet", E_ARG, values=((-2, 0, 2), (0.2, 0.6, 0.2)), shift=2)
    add("all-even alphabet, one value", E_ARG, values=((0,), (1.0,)))
    add("odd value of probability 0", ok, values=((0, 1), (1.0, 0.0)))
    add("six values", ok, values=((-3, -2, -1, 1, 2, 3), (1,) * 6), shift=3)
    return out


def table():
    return [r for S in SIZES + BAD_SIZES for r in _rows(S)]


def _run_table() -> None:
    """Child process: every row's return code, as JSON on stdout."""
    assert os.environ.get("CUDA_VISIBLE_DEVICES") == "", "the table runs only where no device is visible"
    L = _lib.lib()
    print(json.dumps({label: L.tg_demo_gen_gf2(*args) for label, args, _ in table()}))


def test_argument_rules_of_the_mod_2_demo_generator():
    rows = table()
    assert len({r[0] for r in rows}) == len(rows)
    res = subprocess.run([sys.executable, "-c", "from tests.test_gf2_demo_ref import _run_table; _run_table()"], cwd=ROOT,
                         env={**os.environ, "CUDA_VISIBLE_DEVICES": ""}, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr
    got = json.loads(res.stdout.strip().splitlines()[-1])
    wrong = [f"{label}: {got[label]}, want {want}" for label, _, want in rows if got[label] != want]
    assert not wrong, f"{len(wrong)} of {len(rows)} calls:\n" + "\n".join(wrong)
