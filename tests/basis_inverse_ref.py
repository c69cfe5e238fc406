"""References for the inverse triples (include/tensorgame.h tg_invert_bases, tg_invert_bases_gf2).

Over Z the contract is one predicate: M has an integer inverse whose entries all lie in [-128, 127].  inverse_int8 decides
it by Gauss-Jordan elimination over fractions.Fraction, the definition the tests pin everything else to.  inverses_int8
decides it for batches, fast and still exactly: a matrix whose rounded float64 inverse Y passes M Y = I in int64 has Y as
its inverse, and every other matrix is inverted modulo 2^31 - 1 and certified (an inverse mod a prime above 256, lifted
to the symmetric range, is the int8 integer inverse iff its entries fit int8 and M X = I holds exactly).  Over GF(2),
inverse_gf2_or_none wraps gf2_basis_ref.inverse_gf2 with a rank test, so that a singular matrix gives None."""
from fractions import Fraction

import numpy as np

from tests import gf2_basis_ref, gf2_ref

FLAG_SINGULAR = 128


def inverse_int8(M):
    """The integer inverse of the square integer matrix M as int64 if it exists with every entry in [-128, 127], else
    None.  Exact: Gauss-Jordan elimination of [M | I] over the rationals."""
    M = np.asarray(M, dtype=np.int64)
    S = M.shape[0]
    a = [[Fraction(int(v)) for v in row] + [Fraction(int(i == r)) for i in range(S)] for r, row in enumerate(M)]
    for c in range(S):
        piv = next((r for r in range(c, S) if a[r][c] != 0), None)
        if piv is None:
            return None
        a[c], a[piv] = a[piv], a[c]
        p = a[c][c]
        a[c] = [v / p for v in a[c]]
        for r in range(S):
            if r != c and a[r][c] != 0:
                f = a[r][c]
                a[r] = [v - f * w for v, w in zip(a[r], a[c])]
    X = [row[S:] for row in a]
    if any(v.denominator != 1 or not -128 <= v <= 127 for row in X for v in row):
        return None
    return np.array([[int(v) for v in row] for row in X], dtype=np.int64)


P31 = (1 << 31) - 1


def _pow_mod(x, e: int, p: int):
    r = np.ones_like(x)
    while e:
        if e & 1:
            r = r * x % p
        x = x * x % p
        e >>= 1
    return r


def _inverses_mod_p(M, p: int = P31):
    """(K, S, S) integer matrices -> (their inverses mod p as residues (K, S, S), invertible mod p (K,)), by batched
    Gauss-Jordan elimination in int64 (residues below 2^31: products below 2^62)"""
    K, S = M.shape[0], M.shape[-1]
    a = np.concatenate([M % p, np.broadcast_to(np.eye(S, dtype=np.int64), (K, S, S))], axis=2)
    ok = np.ones(K, dtype=bool)
    k = np.arange(K)
    for c in range(S):
        nz = a[:, c:, c] != 0
        ok &= nz.any(1)
        piv = c + np.argmax(nz, axis=1)
        prow = a[k, piv].copy()
        a[k, piv] = a[:, c]
        a[:, c] = prow * _pow_mod(prow[:, c], p - 2, p)[:, None] % p
        f = a[:, :, c].copy()
        f[:, c] = 0
        a = (a - f[:, :, None] * a[:, c][:, None, :] % p) % p
    return a[:, :, S:], ok


def inverses_int8(mats):
    """(N, 3, S, S) integer triples -> (inv int64 (N, 3, S, S), flags uint8 (N,)) as tg_invert_bases writes them: each
    matrix's int8 integer inverse, or zeros and FLAG_SINGULAR on its triple."""
    mats = np.asarray(mats, dtype=np.int64)
    N, S = mats.shape[0], mats.shape[-1]
    flat = mats.reshape(-1, S, S)
    eye = np.eye(S, dtype=np.int64)
    with np.errstate(all="ignore"):
        Y = np.nan_to_num(np.rint(np.linalg.pinv(flat.astype(np.float64))), nan=2.0 ** 50)
    small = (np.abs(Y) <= 2.0 ** 40).all((1, 2))
    X = np.where(small[:, None, None], Y, 0).astype(np.int64)
    certified = small & (flat @ X == eye).all((1, 2))  # |M Y| <= 16 * 128 * 2^40: exact in int64
    rest = np.flatnonzero(~certified)
    if rest.size:
        r, inv_p = _inverses_mod_p(flat[rest])
        r = np.where(r > P31 // 2, r - P31, r)
        fits = inv_p & ((r >= -128) & (r <= 127)).all((1, 2))
        r[~fits] = 0
        X[rest] = r
        certified[rest] = fits & (flat[rest] @ r == eye).all((1, 2))
    ok = certified & ((X >= -128) & (X <= 127)).all((1, 2))
    X[~ok] = 0
    return X.reshape(N, 3, S, S), np.where(ok.reshape(N, 3).all(1), 0, FLAG_SINGULAR).astype(np.uint8)


def inverse_gf2_or_none(M):
    """The inverse over GF(2) of M mod 2 as 0/1 int64, or None where M is singular over GF(2)."""
    M = np.asarray(M, dtype=np.int64) & 1
    if gf2_ref.rank_gf2(M) < M.shape[0]:
        return None
    return gf2_basis_ref.inverse_gf2(M)


def inverses_gf2(bits, S: int):
    """int32 (N, 3, S) bit-matrix triples (bits S to 31 ignored) -> (inv int32 (N, 3, S), flags uint8 (N,)) as
    tg_invert_bases_gf2 writes them: each matrix's inverse, or zero rows and FLAG_SINGULAR on its triple."""
    M = gf2_basis_ref.bits_to_mats(bits, S)
    N = M.shape[0]
    inv = np.zeros_like(M)
    flags = np.zeros(N, dtype=np.uint8)
    for n in range(N):
        for f in range(3):
            X = inverse_gf2_or_none(M[n, f])
            if X is None:
                flags[n] = FLAG_SINGULAR
            else:
                inv[n, f] = X
    return gf2_basis_ref.mats_to_bits(inv), flags


def _chain(S: int, a: int, b: int) -> np.ndarray:
    """I with M[0][1] = a and M[1][2] = b: its inverse has -a, -b and a b above the diagonal"""
    M = np.eye(S, dtype=np.int64)
    M[0, 1], M[1, 2] = a, b
    return M


def _diag(S: int, d) -> np.ndarray:
    return np.diag(list(d) + [1] * (S - len(d))).astype(np.int64)


def mod_p_impostor(S: int) -> np.ndarray:
    """A unimodular int8 matrix whose integer inverse has the entry 127^2 + 127^2 + 7 * 71 = 32755 = 32749 + 6, and every
    other entry in int8: its inverse modulo 32749, lifted to (-p/2, p/2), has only int8 entries (6 in place of 32755) and is
    not its inverse.  Only the exact M X = I check tells the two apart.  I + N with N = x in row 0 (columns 1..3) and y in
    column S-1 (rows 1..3): N^2 has the single entry x . y at (0, S-1) and N^3 = 0, so the inverse is I - N + N^2."""
    M = np.eye(S, dtype=np.int64)
    M[0, 1:4] = (127, 127, 7)
    M[1:4, S - 1] = (127, 127, 71)
    return M


def integer_edges(S: int, rng) -> list:
    """(label, matrix, has an int8 integer inverse) at the edges of tg_invert_bases' predicate"""
    perm = np.eye(S, dtype=np.int64)[rng.permutation(S)] * rng.choice([-1, 1], size=(S, 1))
    self_inverse = np.eye(S, dtype=np.int64)
    self_inverse[0, 0], self_inverse[0, 1] = -1, -128  # [[-1, -128], [0, 1]] is its own inverse
    twin_rows = rng.integers(-3, 4, size=(S, S))
    twin_rows[1] = twin_rows[0]
    det_m1 = _chain(S, 5, -7)
    det_m1[S - 1, S - 1] = -1
    out = [
        ("identity", np.eye(S, dtype=np.int64), True),
        ("signed permutation", perm, True),
        ("inverse entry 127", _chain(S, -127, -1), True),
        ("inverse entry -128", _chain(S, -16, 8), True),
        ("inverse entry 128", _chain(S, 16, 8), False),
        ("inverse entry -129", _chain(S, -3, 43), False),
        ("-128 in a self-inverse matrix", self_inverse, True),
        ("-128 above the diagonal (inverse 128)", _chain(S, -128, 0), False),
        ("-128 on the diagonal", _diag(S, [-128]), False),
        ("det 0: zero row", np.where(np.arange(S)[:, None] == 1, 0, rng.integers(-3, 4, size=(S, S))), False),
        ("det 0: two equal rows", twin_rows, False),
        ("det 2", _diag(S, [2]), False),
        ("det -1", det_m1, True),
        ("det 4 * 32749 - 1", _diag(S, [123, 71, 15]), False),
        ("det 11 * 32749 + 1", _diag(S, [120, 79, 38]), False),
    ]
    if S >= 5:
        out += [("inverse mod 32749 in int8, not the inverse", mod_p_impostor(S), False)]
    if S >= 7:
        out += [("det 2^31", _diag(S, [-128, -128, -128, -128, 2, 2, 2]), False),
                ("det -2^31", _diag(S, [-128, -128, -128, -128, -2, 2, 2]), False)]
    return out
