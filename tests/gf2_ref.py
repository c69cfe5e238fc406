"""numpy references for the mod-2 game path (include/tensorgame.h "mod-2 game path"): the bit slab format, pack / unpack,
step, rollout and replay, state keys and slice rank over GF(2).  States are 0/1 arrays (B,S,S,S); a token t stands for
the coefficient t - shift, whose residue is (t - shift) & 1."""
import numpy as np

from tests import i16_ref

FLAG_TERMINAL, FLAG_NULL = 1, 2


def geo(S: int):
    """(RW words per row, GB bytes per game)"""
    rw = (S * S + 31) // 32
    return rw, (4 * S * rw + 15) & ~15


def dense_to_bits(T) -> np.ndarray:
    """(B,S,S,S) integers -> bit slab int32 (B, GB/4) of their residues mod 2 (low bit of the two's complement)."""
    T = np.asarray(T, dtype=np.int64) & 1
    B, S = T.shape[0], T.shape[-1]
    rw, gb = geo(S)
    rows = np.zeros((B, S, 32 * rw), dtype=np.uint64)
    rows[:, :, : S * S] = T.reshape(B, S, S * S)
    words = (rows.reshape(B, S, rw, 32) << np.arange(32, dtype=np.uint64)).sum(-1, dtype=np.uint64)
    out = np.zeros((B, gb // 4), dtype=np.uint32)
    out[:, : S * rw] = words.reshape(B, S * rw).astype(np.uint32)
    return out.view(np.int32)


def bits_to_dense(bits, S: int) -> np.ndarray:
    """bit slab (B, GB/4) -> 0/1 int64 (B,S,S,S); asserts padding bits and words are zero."""
    bits = np.ascontiguousarray(bits).view(np.uint32)
    B = bits.shape[0]
    rw, gb = geo(S)
    assert bits.shape[1] == gb // 4
    assert not bits[:, S * rw :].any(), "padding words must be zero"
    w = bits[:, : S * rw].reshape(B, S, rw).astype(np.uint64)
    b = ((w[..., None] >> np.arange(32, dtype=np.uint64)) & 1).reshape(B, S, 32 * rw)
    assert not b[:, :, S * S :].any(), "padding bits must be zero"
    return b[:, :, : S * S].reshape(B, S, S, S).astype(np.int64)


def factors_mod2(tok, shift: int):
    tok = np.asarray(tok, dtype=np.int64)
    S = tok.shape[-1] // 3
    return [(tok[..., m * S:(m + 1) * S] - shift) & 1 for m in range(3)]


def rank1(tok, shift: int) -> np.ndarray:
    """tok (..., 3S) -> (..., S, S, S) 0/1: u (x) v (x) w mod 2."""
    u, v, w = factors_mod2(tok, shift)
    return u[..., :, None, None] & v[..., None, :, None] & w[..., None, None, :]


def step_ref(T, tok, shift: int):
    """T (B,S,S,S) 0/1, tok (B,3S) -> (T xor rank1, flags, nnz)."""
    T = np.asarray(T, dtype=np.int64) & 1
    B = T.shape[0]
    out = T ^ rank1(tok, shift)
    u, v, w = factors_mod2(tok, shift)
    null = ~(u.any(-1) & v.any(-1) & w.any(-1))
    flags = np.where(~out.reshape(B, -1).any(1), FLAG_TERMINAL, 0) | np.where(null, FLAG_NULL, 0)
    return out, flags.astype(np.uint8), np.count_nonzero(out.reshape(B, -1), axis=1).astype(np.int32)


def rollout_ref(T, tape, shift: int, freeze: bool = True):
    """T (B,S,S,S) 0/1, tape (B,K,3S) -> (T_out, flags, nnz, steps); with freeze a game stops at its first all-zero
    state (steps = actions applied), without it all K actions are applied."""
    cur = np.asarray(T, dtype=np.int64) & 1
    tape = np.asarray(tape, dtype=np.int64)
    B, K = cur.shape[0], tape.shape[1]
    alive = cur.reshape(B, -1).any(1) if freeze else np.ones(B, dtype=bool)
    steps = np.zeros(B, dtype=np.int32)
    for t in range(K):
        cur[alive] ^= rank1(tape[alive, t], shift)
        steps[alive] = t + 1
        if freeze:
            alive &= cur.reshape(B, -1).any(1)
    nnz = np.count_nonzero(cur.reshape(B, -1), axis=1).astype(np.int32)
    return cur, np.where(nnz == 0, FLAG_TERMINAL, 0).astype(np.uint8), nnz, steps


def state_keys(T) -> np.ndarray:
    """tg_state_key of the 0/1 values (the trilinear form of tests/i16_ref.py)."""
    return i16_ref.state_keys(np.asarray(T, dtype=np.int64) & 1)


def rank_gf2(M) -> int:
    """rank over GF(2) of an integer matrix (entries taken mod 2), by elimination on Python-integer rows."""
    rows = [int("".join(str(int(x) & 1) for x in r[::-1]), 2) for r in np.asarray(M)]
    rank = 0
    for c in range(np.asarray(M).shape[1]):
        piv = next((i for i in range(rank, len(rows)) if (rows[i] >> c) & 1), None)
        if piv is None:
            continue
        rows[rank], rows[piv] = rows[piv], rows[rank]
        for i in range(len(rows)):
            if i != rank and (rows[i] >> c) & 1:
                rows[i] ^= rows[rank]
        rank += 1
    return rank


def slice_ranks(T) -> np.ndarray:
    """sum_i rank_GF(2)(T[b,i,:,:]) per game."""
    T = np.asarray(T)
    return np.array([sum(rank_gf2(t[i]) for i in range(t.shape[0])) for t in T], dtype=np.int32)


def random_invertible(S: int, rng) -> np.ndarray:
    """A random S x S matrix invertible over GF(2) (resampled until it is)."""
    while True:
        M = rng.integers(0, 2, size=(S, S))
        if rank_gf2(M) == S:
            return M


def with_rank(S: int, r: int, rng) -> np.ndarray:
    """P diag(1^r, 0^(S-r)) Q mod 2 for random invertible P, Q: an S x S matrix of rank exactly r over GF(2)."""
    D = np.zeros((S, S), dtype=np.int64)
    D[np.arange(r), np.arange(r)] = 1
    return (random_invertible(S, rng) @ D @ random_invertible(S, rng)) & 1
