"""Exact references for the edge tests of tests/test_edges_gpu.py, and checks of those references.

The kernels work in packed or reduced arithmetic that is exact only inside hand-derived bounds (int8 offset binary,
16-bit lanes, f16 operands, int32 accumulators, arithmetic mod 2^31 - 1).  The references here use int64 numpy or
Python integers, so they hold at and beyond every such bound; the edge tests construct inputs on both sides of each
bound and compare the kernels with them."""
import numpy as np
import pytest

from oracle import tg_oracle as orc

P31 = 2**31 - 1
# an int8 4x4 matrix with det = 2^31 - 1: rank 4 over Q, rank 3 over GF(2^31 - 1)
DET_P = [[71, 119, 113, 101], [95, -119, 101, -126], [125, 98, -113, -128], [99, -120, -100, 103]]


def det_int(M) -> int:
    """Determinant over Z (Bareiss, Python integers)."""
    M = [[int(x) for x in row] for row in M]
    n, sign, prev = len(M), 1, 1
    for k in range(n - 1):
        if M[k][k] == 0:
            swap = next((i for i in range(k + 1, n) if M[i][k] != 0), None)
            if swap is None:
                return 0
            M[k], M[swap], sign = M[swap], M[k], -sign
        for i in range(k + 1, n):
            for j in range(k + 1, n):
                M[i][j] = (M[i][j] * M[k][k] - M[i][k] * M[k][j]) // prev
        prev = M[k][k]
    return sign * M[n - 1][n - 1]


def rank_int(M) -> int:
    """Rank over Q (Bareiss fraction-free echelon form, Python integers; every division is exact)."""
    rows = [[int(x) for x in row] for row in M]
    rank, prev = 0, 1
    for c in range(len(rows[0]) if rows else 0):
        piv = next((i for i in range(rank, len(rows)) if rows[i][c] != 0), None)
        if piv is None:
            continue
        rows[rank], rows[piv] = rows[piv], rows[rank]
        p = rows[rank]
        for i in range(rank + 1, len(rows)):
            f = rows[i][c]
            rows[i] = [(p[c] * x - f * y) // prev for x, y in zip(rows[i], p)]
        prev, rank = p[c], rank + 1
    return rank


def slice_ranks(T) -> np.ndarray:
    """sum over i of rank_Q(T[b, i]) for (B,S,S,S) integers."""
    return np.array([sum(rank_int(t[i]) for i in range(t.shape[0])) for t in np.asarray(T)], dtype=np.int64)


def change_of_basis_ref(T, A, Bm, Cm) -> np.ndarray:
    """T'[i,j,k] = sum_abc A[i,a] B[j,b] C[k,c] T[a,b,c] in int64 (|T'| <= S^3 2^28 < 2^63)."""
    T, A, Bm, Cm = (np.asarray(x, dtype=np.int64) for x in (T, A, Bm, Cm))
    return np.einsum("ia,jb,kc,abc->ijk", A, Bm, Cm, T, optimize=True)


def rank1_sum(tok, shift) -> np.ndarray:
    """tok (N,R,3S) token values -> (N,S,S,S) int64 sum_r u_r (x) v_r (x) w_r, coefficient = token - shift."""
    tok = np.asarray(tok, dtype=np.int64)
    S = tok.shape[-1] // 3
    u, v, w = (tok[..., m * S:(m + 1) * S] - shift for m in range(3))
    return np.einsum("nri,nrj,nrk->nijk", u, v, w)


def basis_counterexample(S: int):
    """A game and matrices whose T' is exactly 2^32 in every entry (wraps to 0 in int32)."""
    T = np.zeros((S, S, S), dtype=np.int64)
    T[0:2, 0:2, 0:4] = -128
    A = np.zeros((S, S), dtype=np.int64)
    A[:, 0:2] = -128
    Cm = np.zeros((S, S), dtype=np.int64)
    Cm[:, 0:4] = -128
    return T, A, A.copy(), Cm


def block_diag_det_p(S: int) -> np.ndarray:
    """An S x S int8 matrix with floor(S/4) copies of DET_P on the diagonal: rank_Q = 4 floor(S/4), while
    GF(2^31 - 1) sees one rank less per copy."""
    M = np.zeros((S, S), dtype=np.int64)
    for q in range(S // 4):
        M[4 * q:4 * q + 4, 4 * q:4 * q + 4] = DET_P
    return M


def test_det_p_matrix_is_full_rank_over_q_and_singular_mod_p():
    assert det_int(DET_P) == P31
    assert rank_int(DET_P) == 4
    assert np.linalg.matrix_rank(np.array(DET_P, dtype=np.float32)) == 4
    # rank mod p is 3: the matrix reduced mod p has a vanishing determinant
    assert det_int(DET_P) % P31 == 0


@pytest.mark.parametrize("S", [4, 9, 16, 25])
def test_block_diag_rank(S):
    M = block_diag_det_p(S)
    assert rank_int(M) == 4 * (S // 4)
    assert np.linalg.matrix_rank(M.astype(np.float64)) == 4 * (S // 4)


def test_rank_int_against_numpy_and_oracle():
    rng = np.random.default_rng(0)
    for S in (4, 9, 16):
        T = rng.integers(-3, 4, size=(6, S, S, S))
        T[:, :, :, S // 2] = 0  # rank-deficient slices too
        T[1, 2] = np.outer(rng.integers(-3, 4, S), rng.integers(-3, 4, S))
        want = np.array([sum(np.linalg.matrix_rank(t[i].astype(np.float64)) for i in range(S)) for t in T])
        assert np.array_equal(slice_ranks(T), want)
        assert np.array_equal(orc.slice_rank_batch(T), want)
    # the oracle (mod 2^61 - 1) gets the det = 2^31 - 1 slice right
    T = np.zeros((1, 4, 4, 4), dtype=np.int64)
    T[0, 0] = DET_P
    assert orc.slice_rank_batch(T)[0] == 4 == slice_ranks(T)[0]


def test_rank_int_full_range_against_float64():
    rng = np.random.default_rng(3)
    for n in (4, 9, 16, 25):
        for r in (1, n // 2, n - 1, n):
            M = rng.integers(-128, 128, size=(n, r)) @ rng.integers(-1, 2, size=(r, n))
            M = np.clip(M, -128, 127) if r == 1 else M
            assert rank_int(M) == np.linalg.matrix_rank(M.astype(np.float64))


def test_det_int_and_rank_int_small_cases():
    assert det_int([[0, 1], [1, 0]]) == -1
    assert det_int([[2, 3], [4, 6]]) == 0
    assert rank_int([[2, 3], [4, 6]]) == 1
    assert rank_int([[0, 0], [0, 0]]) == 0
    assert det_int([[-128] * 3, [0, -128, 0], [0, 0, 127]]) == -128 * -128 * 127


@pytest.mark.parametrize("S", [4, 9, 16])
def test_change_of_basis_counterexample_is_2_pow_32(S):
    T, A, Bm, Cm = basis_counterexample(S)
    ref = change_of_basis_ref(T, A, Bm, Cm)
    assert (ref == 2**32).all()
    assert ((ref.astype(np.int64) & 0xFFFFFFFF) == 0).all()  # what an int32 accumulator would hold
    assert np.array_equal(ref, orc.change_of_basis(T, A, Bm, Cm))


@pytest.mark.parametrize("S", [4, 9, 16])
def test_change_of_basis_ref_matches_oracle(S):
    rng = np.random.default_rng(S)
    T = rng.integers(-128, 128, size=(S, S, S))
    A, Bm, Cm = (rng.integers(-128, 128, size=(S, S)) for _ in range(3))
    assert np.array_equal(change_of_basis_ref(T, A, Bm, Cm), orc.change_of_basis(T, A, Bm, Cm))


def test_accumulate_i16_counterexample_is_2_pow_32():
    S, R = 4, 2048
    tok = np.zeros((1, R, 3 * S), dtype=np.int64)
    tok[:, :, [0, S, 2 * S]] = 128
    ref = rank1_sum(tok, 0)
    assert ref[0, 0, 0, 0] == 2**32 and np.count_nonzero(ref) == 1
    tok[:] = 127
    tok[:, :, [0, S, 2 * S]] = 255
    assert rank1_sum(tok, 127)[0, 0, 0, 0] == 2**32 and np.count_nonzero(rank1_sum(tok, 127)) == 1
    # the first tape length whose terms can carry an int32 sum past 2^31 at shift 0
    assert 129 * 255**3 < 2**31 <= 130 * 255**3


@pytest.mark.parametrize("S", [4, 9])
def test_rank1_sum_matches_oracle(S):
    rng = np.random.default_rng(7)
    tok = rng.integers(0, 9, size=(3, 5, 3 * S))
    want = np.stack([sum(orc.action_to_tensor(t, 4).astype(np.int64) for t in d) for d in tok])
    assert np.array_equal(rank1_sum(tok, 4), want)
