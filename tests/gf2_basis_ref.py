"""numpy references for the change of basis over GF(2) (include/tensorgame.h "change of basis mod 2"): bit matrices, the
tensor transform one mode at a time, the factor transform, the invertible sampler restated from the Philox stream, and
inversion over GF(2).  Matrices are 0/1 (or integer) arrays (..., 3, S, S) = (A, B, C); states are (N, S, S, S)."""
import numpy as np

from tests import oracle_any_s as orx

PHILOX_MATS = 0x6D617473  # third counter word of the matrix draws (orc_sample_unimodular)


def mats_to_bits(M) -> np.ndarray:
    """(..., 3, S, S) integers -> int32 (..., 3, S) bit matrices of their residues: word r of a matrix is row r, bit c
    entry (r, c) mod 2."""
    M = np.asarray(M, dtype=np.int64) & 1
    S = M.shape[-1]
    return (M << np.arange(S, dtype=np.int64)).sum(-1).astype(np.uint32).view(np.int32)


def bits_to_mats(bits, S: int) -> np.ndarray:
    """int32 (..., 3, S) bit matrices -> 0/1 int64 (..., 3, S, S); bits S to 31 of a row are ignored."""
    w = np.asarray(bits).astype(np.int64) & 0xFFFFFFFF
    return (w[..., None] >> np.arange(S, dtype=np.int64)) & 1


def transform(T, M) -> np.ndarray:
    """T' = T x1 A x2 B x3 C mod 2 in int64, one mode at a time with mod 2 after each.  T (N, S, S, S) integers, M
    (N or 1, 3, S, S) integers -> 0/1 int64 (N, S, S, S)."""
    T = np.asarray(T, dtype=np.int64) & 1
    M = np.asarray(M, dtype=np.int64) & 1
    A, B, C = (np.broadcast_to(M[:, f], (T.shape[0],) + M.shape[2:]) for f in range(3))
    N, S = T.shape[0], T.shape[-1]
    T = np.matmul(A, T.reshape(N, S, S * S)).reshape(N, S, S, S) & 1                  # mode 1: i <- a
    T = np.matmul(B[:, None], T) & 1                                                  # mode 2: j <- b
    T = np.matmul(T, np.swapaxes(C, -1, -2)[:, None]) & 1                            # mode 3: k <- c
    return T


def factors(tok, M, shift_in: int, shift_out: int) -> np.ndarray:
    """Tokens (N, R, 3S) of residues (t - shift_in) & 1 -> tokens (N, R, 3S) of u' = A u, v' = B v, w' = C w mod 2 plus
    shift_out.  M (N or 1, 3, S, S)."""
    tok = np.asarray(tok, dtype=np.int64)
    M = np.asarray(M, dtype=np.int64) & 1
    N, R, S = tok.shape[0], tok.shape[1], tok.shape[2] // 3
    x = ((tok - shift_in) & 1).reshape(N, R, 3, S)
    M = np.broadcast_to(M, (N, 3, S, S))
    y = np.einsum("nfia,nrfa->nrfi", M, x) & 1
    return y.reshape(N, R, 3 * S) + shift_out


def rank1_sum(tok, shift: int) -> np.ndarray:
    """sum_r u_r (x) v_r (x) w_r mod 2 of tokens (N, R, 3S) -> 0/1 (N, S, S, S)."""
    x = (np.asarray(tok, dtype=np.int64) - shift) & 1
    S = x.shape[-1] // 3
    return np.einsum("nri,nrj,nrk->nijk", x[..., :S], x[..., S:2 * S], x[..., 2 * S:]) & 1


def sample_invertible(seed: int, first: int, n: int, S: int, p_nonzero: float) -> np.ndarray:
    """The sampler contract for any S -> 0/1 int64 (n, 3, S, S): entry e = r S + c of matrix f of game d = first + i
    draws byte e % 16 of Philox block e // 16 with counter (block, f, 0x6D617473, d_lo) and key (seed_lo ^ d_hi *
    0x9E3779B9, seed_hi); the draw is non-zero iff its low 7 bits are below floor(128 p).  L = the non-zero draws below
    the diagonal plus I, U = those above it plus I, M = L U mod 2."""
    thr = int(p_nonzero * 128.0)
    nb = (S * S + 15) // 16
    e = np.arange(S * S)
    out = np.zeros((n, 3, S, S), dtype=np.int64)
    eye = np.eye(S, dtype=np.int64)
    for i in range(n):
        d = first + i
        k0 = (seed & 0xFFFFFFFF) ^ (((d >> 32) * 0x9E3779B9) & 0xFFFFFFFF)
        blk = orx.philox4x32_10(np.tile(np.arange(nb, dtype=np.uint32), 3), np.repeat(np.arange(3, dtype=np.uint32), nb),
                                np.full(3 * nb, PHILOX_MATS, dtype=np.uint32), np.full(3 * nb, d & 0xFFFFFFFF, dtype=np.uint32),
                                k0, (seed >> 32) & 0xFFFFFFFF)
        words = np.stack(blk, axis=1).astype(np.int64).reshape(3, nb, 4)  # [f][block][word]
        for f in range(3):
            byte = (words[f, e >> 4, (e >> 2) & 3] >> (8 * (e & 3))) & 0xFF
            nz = ((byte & 0x7F) < thr).astype(np.int64).reshape(S, S)
            L, U = np.tril(nz, -1) + eye, np.triu(nz, 1) + eye
            out[i, f] = (L @ U) & 1
    return out


def inverse_gf2(M) -> np.ndarray:
    """Inverse over GF(2) of an invertible S x S matrix (entries taken mod 2), by Gauss-Jordan elimination."""
    M = np.asarray(M, dtype=np.int64) & 1
    S = M.shape[0]
    a = np.concatenate([M, np.eye(S, dtype=np.int64)], axis=1)
    for c in range(S):
        piv = c + int(np.argmax(a[c:, c]))
        assert a[piv, c], "matrix is singular over GF(2)"
        a[[c, piv]] = a[[piv, c]]
        rows = np.nonzero(a[:, c])[0]
        rows = rows[rows != c]
        a[rows] ^= a[c]
    return a[:, S:]
