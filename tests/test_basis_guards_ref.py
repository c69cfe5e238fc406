"""The change of basis's guard model (tests/basis_guard_ref.py) and its edge cases, on the CPU: every case sits where it
claims (its intermediate values, bounds and path), and the exact reference agrees with the C oracle on every case."""
import numpy as np
import pytest

from oracle import tg_oracle as orc
from tests import basis_guard_ref as gr
from tests.test_edges_ref import change_of_basis_ref

CASES = gr.all_cases()


@pytest.mark.parametrize("case", CASES, ids=lambda c: c.name)
def test_case_sits_where_it_claims(case):
    for M in (case.T, case.A, case.B, case.C):
        assert M.min() >= -128 and M.max() <= 127  # every input is int8
    g = gr.model(case.T, case.A, case.B, case.C, case.out, case.align)
    have = {**vars(g), **gr.derived(g)}
    for key, want in case.claims.items():
        assert have[key] == want, (key, have[key], want)


@pytest.mark.parametrize("case", CASES, ids=lambda c: c.name)
def test_reference_matches_oracle(case):
    assert np.array_equal(change_of_basis_ref(case.T, case.A, case.B, case.C),
                          orc.change_of_basis(case.T, case.A, case.B, case.C))


def test_every_path_and_both_sides_are_covered():
    paths = {(c.S, gr.model(c.T, c.A, c.B, c.C, c.out, c.align).path) for c in CASES}
    assert paths == {(16, "f16_apriori"), (16, "f16_checked"), (16, "planes"), (16, "exact"), (9, "f16_apriori"),
                     (9, "f16_tracked"), (9, "exact"), (4, "lanes"), (4, "exact")}
    # each threshold with a case on the accepting side (== the constant) and on the rejecting side
    d = [gr.derived(gr.model(c.T, c.A, c.B, c.C, c.out, c.align)) for c in CASES]
    for key, at in (("yb", 2047), ("zb", 2047), ("maxY", 2047), ("maxZ", 2047), ("maxZ*nA", 32752),
                    ("ybound*nA*nB", 32512), ("tb*nC*nB*nA", 32640), ("maxY*nA*nB", 32767)):
        assert any(x[key] == at for x in d), key
        assert any(x[key] > gr.BITS16_MAX if at > 2047 else x[key] == 2048 for x in d), key


def test_model_helpers():
    assert gr.or_bound([1, 2]) == 4 and gr.or_bound(np.full(5, -23)) == 23 and gr.or_bound([-128, 127]) == 128
    assert gr.or_bound([0]) == 1
    assert list(gr.hi8([-256, -1, 255, 256, -16256, 16256, 32767, -32768])) == [-1, -1, 0, 1, -64, 63, 127, -128]
    assert gr.norm([[1, -2], [-128, 0]]) == 128
    # |Y| <= 256 (mag(hi8) + 1) whenever Y fits 16 bits
    y = np.arange(-32768, 32768)
    assert (np.abs(y) <= 256 * (gr.mag(gr.hi8(y)) + 1)).all()


@pytest.mark.parametrize("out", ["int8", "int16"])
def test_model_flags_on_random_games(out):
    """Identity matrices keep every game on the cheapest path; RANGE is exactly 'T' leaves the output's zone'."""
    rng = np.random.default_rng(5)
    for S, fast in ((4, "thread"), (9, "f16_apriori"), (16, "f16_apriori")):
        for _ in range(4):
            T = rng.integers(-128, 128, (S, S, S))
            I = np.eye(S, dtype=np.int64)
            g = gr.model(T, I, I, I, out)
            assert g.path == fast and np.array_equal(g.ref, T)
            lo, hi = gr.ZONE[out]
            assert g.flags == (gr.RANGE if ((T < lo) | (T > hi)).any() else 0)
    # unaligned mats route 16x16x16 to the exact kernel and 4x4x4 to the packed lanes
    T = np.zeros((16,) * 3, dtype=np.int64)
    assert gr.model(T, *[np.eye(16, dtype=np.int64)] * 3, out, align=2).flags == gr.PATH_EXACT
    assert gr.model(np.zeros((4,) * 3), *[np.eye(4, dtype=np.int64)] * 3, out, align=4).path == "lanes"
