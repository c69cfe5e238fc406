"""Exact references for the int16 game path (tg_step_i16, tg_expand_children_i16, tg_rollout_i16, tg_replay_i16,
tg_state_key_i16, tg_slice_rank_i16): int64 numpy and Python integers, so they hold at and beyond every bound of the
kernels' packed 16-bit arithmetic.  Contract (include/tensorgame.h "int16 game path"): entries are guaranteed while they
stay in [-16384, 16383]; a result outside that zone, or a token above 2 * shift, raises FLAG_RANGE."""
import numpy as np

FLAG_TERMINAL, FLAG_NULL, FLAG_RANGE = 1, 2, 4
ZONE_LO, ZONE_HI = -16384, 16383
M64 = (1 << 64) - 1


def geo(S: int):
    rp = (S * S + 3) & ~3
    return rp, (S * rp + 15) & ~15, (3 * S + 15) & ~15


def dense_to_slab16(T) -> np.ndarray:
    """(B,S,S,S) integers in int16 -> int16 slab (B,GP), padding zero."""
    T = np.asarray(T)
    B, S = T.shape[0], T.shape[-1]
    rp, gp, _ = geo(S)
    assert T.min(initial=0) >= -32768 and T.max(initial=0) <= 32767
    slab = np.zeros((B, gp), dtype=np.int16)
    slab[:, : S * rp].reshape(B, S, rp)[:, :, : S * S] = T.reshape(B, S, S * S)
    return slab


def slab16_to_dense(slab, S: int) -> np.ndarray:
    """int16 slab (B,GP) -> int64 (B,S,S,S); asserts the padding is zero."""
    slab = np.asarray(slab)
    B = slab.shape[0]
    rp, gp, _ = geo(S)
    assert slab.shape[1] == gp
    rows = slab[:, : S * rp].reshape(B, S, rp)
    assert not rows[:, :, S * S :].any() and not slab[:, S * rp :].any(), "slab padding must stay zero"
    return rows[:, :, : S * S].reshape(B, S, S, S).astype(np.int64)


def rank1(tok, shift: int) -> np.ndarray:
    """tok (..., 3S) tokens -> (..., S, S, S) int64 u (x) v (x) w with coefficient = token - shift."""
    tok = np.asarray(tok, dtype=np.int64)
    S = tok.shape[-1] // 3
    u, v, w = (tok[..., m * S:(m + 1) * S] - shift for m in range(3))
    return u[..., :, None, None] * v[..., None, :, None] * w[..., None, None, :]


def outside(T) -> np.ndarray:
    """per game: an entry outside [-16384, 16383]"""
    T = np.asarray(T)
    return ((T < ZONE_LO) | (T > ZONE_HI)).reshape(T.shape[0], -1).any(1)


def over_bound(tok, shift: int) -> np.ndarray:
    """per record: a token above 2 * shift"""
    return (np.asarray(tok) > 2 * shift).any(-1)


def step_ref(T, tok, shift: int):
    """T (B,S,S,S), tok (B,3S) -> (T - rank1, flags, nnz) under the int16 contract."""
    T = np.asarray(T, dtype=np.int64)
    d = rank1(tok, shift)
    out = T - d
    B = T.shape[0]
    flags = np.where(~out.reshape(B, -1).any(1), FLAG_TERMINAL, 0)
    flags |= np.where(~d.reshape(B, -1).any(1), FLAG_NULL, 0)
    flags |= np.where(outside(out) | over_bound(tok, shift), FLAG_RANGE, 0)
    return out, flags.astype(np.uint8), np.count_nonzero(out.reshape(B, -1), axis=1).astype(np.int32)


def rollout_ref(T, tape, shift: int, freeze: bool = True):
    """T (B,S,S,S), tape (B,K,3S) -> (T_out, flags, nnz, steps): K steps, a game frozen at its first all-zero state
    when freeze; RANGE = the start state or the state after an applied step left the zone, or an applied step's
    record broke the token bound."""
    cur = np.array(T, dtype=np.int64)
    tape = np.asarray(tape, dtype=np.int64)
    B, K = cur.shape[0], tape.shape[1]
    bad = outside(cur)
    alive = cur.reshape(B, -1).any(1) if freeze else np.ones(B, dtype=bool)
    steps = np.zeros(B, dtype=np.int32)
    for t in range(K):
        if not alive.any():
            break
        a = alive
        cur[a] -= rank1(tape[a, t], shift)
        steps[a] = t + 1
        bad[a] |= outside(cur[a]) | over_bound(tape[a, t], shift)
        if freeze:
            alive = a & cur.reshape(B, -1).any(1)
    nz = cur.reshape(B, -1).any(1)
    flags = np.where(~nz, FLAG_TERMINAL, 0) | np.where(bad, FLAG_RANGE, 0)
    return cur, flags.astype(np.uint8), np.count_nonzero(cur.reshape(B, -1), axis=1).astype(np.int32), steps


def splitmix64(z: int) -> int:
    z = (z + 0x9E3779B97F4A7C15) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def key_consts(S: int):
    """A_i, B_j, C_k of the state key: splitmix64(0x1000 / 0x2000 / 0x3000 + index) | 1"""
    return [[splitmix64(base + i) | 1 for i in range(S)] for base in (0x1000, 0x2000, 0x3000)]


def state_key_int(T) -> int:
    """key(T) = sum T[i][j][k] A_i B_j C_k mod 2^64 in Python integers, one (S,S,S) state."""
    T = np.asarray(T)
    A, Bc, Cc = key_consts(T.shape[-1])
    total = 0
    for i, a in enumerate(A):
        for j, b in enumerate(Bc):
            total += a * b * sum(int(x) * c for x, c in zip(T[i, j], Cc))
    return total & M64


def state_keys(T) -> np.ndarray:
    """state_key_int of a batch (B,S,S,S), in uint64 numpy arithmetic (wraps mod 2^64 like the formula)."""
    T = np.asarray(T, dtype=np.int64)
    A, Bc, Cc = (np.array(x, dtype=np.uint64) for x in key_consts(T.shape[-1]))
    coef = A[:, None, None] * Bc[None, :, None] * Cc[None, None, :]
    with np.errstate(over="ignore"):
        return (T.astype(np.uint64) * coef).reshape(T.shape[0], -1).sum(1, dtype=np.uint64)


def companion_det(n: int) -> np.ndarray:
    """A 4x4 int16 matrix with determinant n for 2^31 - 2^17 <= n <= 2^31 + 2^16:
    [[1,0,0,a],[0,1,0,b],[0,0,1,c],[x,y,w,z]] has det z - a x - b y - c w."""
    a = b = 32767
    x = y = -32767
    rest = n - 2 * 32767 * 32767  # = z - c w
    c, w = 4, -((rest - 1) // 4)
    z = rest + c * w
    M = np.array([[1, 0, 0, a], [0, 1, 0, b], [0, 0, 1, c], [x, y, w, z]], dtype=np.int64)
    assert np.abs(M).max() <= 32767
    return M
