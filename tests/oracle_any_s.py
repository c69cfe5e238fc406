"""numpy restatement of the oracle functions whose C versions (oracle/tg_oracle.c) keep one game's scratch tensors in
fixed 4096-entry stack buffers, i.e. hold S <= 16 only: the K-step rollout, the training-sample item, the throughput
demo contract v1 and the reference's rejection loop on a uniform stream.  Every other oracle function (step, rank-1
tensor, slice rank, state key, matmul tensor, Philox block, thresholds, categorical CDF, MT19937 stream) has no size
limit and is used as is.  tests/test_s25_oracle.py pins this module to the C oracle at 4, 9 and 16 and restates it
independently at 25.  Test infrastructure only."""
from __future__ import annotations

import numpy as np

from oracle import tg_oracle as orc


def rank1(tok, shift: int) -> np.ndarray:
    """(3S,) tokens -> int64 (S,S,S) u (x) v (x) w with coefficient = token - shift (utils.py:56-96)."""
    tok = np.asarray(tok, dtype=np.int64)
    S = tok.shape[-1] // 3
    u, v, w = tok[:S] - shift, tok[S:2 * S] - shift, tok[2 * S:] - shift
    return np.einsum("i,j,k->ijk", u, v, w)


def rollout_batch(T, tape, shift: int):
    """orc_rollout: T (B,S,S,S), tape (B,K,3S) -> (T_out, flags, nnz, steps); a game freezes once its head is all zero
    (act.py:49), steps = actions applied."""
    T = np.asarray(T, dtype=np.int32)
    tape = np.asarray(tape, dtype=np.int32)
    B, K = T.shape[0], tape.shape[1]
    out = T.copy()
    nnz = (out != 0).reshape(B, -1).sum(1).astype(np.int32)
    alive = nnz != 0
    steps = np.zeros(B, dtype=np.int32)
    for t in range(K):
        if not alive.any():
            break
        idx = np.nonzero(alive)[0]
        nxt, fl, nz = orc.step_batch(out[idx], tape[idx, t], shift)
        out[idx], nnz[idx] = nxt, nz
        steps[idx] += 1
        alive[idx] = nz != 0
    flags = (nnz == 0).astype(np.uint32) * orc.FLAG_TERMINAL
    return out, flags, nnz, steps


def demo_getitem(tokens, target, dim_t: int, idx_action: int, replay_shift: int = 1):
    """orc_demo_getitem (datasets.py:77-122): slot 0 = target minus the actions after idx_action, slots 1.. = the rank-1
    tensors of actions min(idx+dim_t-1, R-1) .. idx+1, zero padded."""
    tokens = np.asarray(tokens, dtype=np.int32)
    target = np.asarray(target, dtype=np.int64)
    R, S = tokens.shape[0], target.shape[-1]
    state = np.zeros((dim_t, S, S, S), dtype=np.int64)
    state[0] = target
    for a in range(idx_action + 1, R):
        state[0] -= rank1(tokens[a], replay_shift)
    hi = min(idx_action + dim_t, R)
    for slot, a in enumerate(range(hi - 1, idx_action, -1), start=1):
        state[slot] = rank1(tokens[a], replay_shift)
    return state.astype(np.int32), float(R - idx_action), tokens[idx_action].copy(), -float(idx_action + 1)


# ---------------------------------------------------------------- throughput contract v1 (orc_demo_philox)
_M0, _M1, _W0, _W1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), np.uint32(0x9E3779B9), np.uint32(0xBB67AE85)


def philox4x32_10(c0, c1, c2, c3, k0: int, k1: int):
    """Philox4x32-10 on arrays of counters (uint32), one key."""
    c = [np.asarray(x, dtype=np.uint32) for x in (c0, c1, c2, c3)]
    k0, k1 = np.uint32(k0), np.uint32(k1)
    m32 = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0 = _M0 * c[0].astype(np.uint64)
        p1 = _M1 * c[2].astype(np.uint64)
        c = [((p1 >> np.uint64(32)).astype(np.uint32) ^ c[1] ^ k0), (p1 & m32).astype(np.uint32),
             ((p0 >> np.uint64(32)).astype(np.uint32) ^ c[3] ^ k1), (p0 & m32).astype(np.uint32)]
        k0 = np.uint32((int(k0) + int(_W0)) & 0xFFFFFFFF)
        k1 = np.uint32((int(k1) + int(_W1)) & 0xFFFFFFFF)
    return c


def demos_philox_v1(seed: int, d0: int, n: int, values, probs, R: int, S: int, shift: int, max_tries: int = 64):
    """orc_demo_philox: demo d, term r, try t draws its 3S 15-bit values from Philox block q // 8 with counter
    (d_lo, d_hi, r | t << 16, q // 8) and key (seed_lo, seed_hi); value = first i < n-1 with x < thr[i], else n-1; a try
    is rejected iff u, v or w is all zero; after max_tries the term is the unit triple values[n-1] e_0.
    -> (tokens (n,R,3S), targets (n,S,S,S), exhausted)."""
    values = np.asarray(values, dtype=np.int64)
    thr = orc.philox_thresholds(probs).astype(np.int64)
    nv = len(values)
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    d = (d0 + np.repeat(np.arange(n, dtype=np.uint64), R)).astype(np.uint64)
    r = np.tile(np.arange(R, dtype=np.uint32), n)
    P = n * R
    fac = np.empty((P, 3 * S), dtype=np.int64)
    pending = np.ones(P, dtype=bool)
    q = np.arange(3 * S)
    for t in range(max_tries):
        idx = np.nonzero(pending)[0]
        if idx.size == 0:
            break
        draws = np.empty((idx.size, 3 * S), dtype=np.int64)
        for bq in range((3 * S + 7) // 8):
            blk = philox4x32_10((d[idx] & np.uint64(0xFFFFFFFF)).astype(np.uint32), (d[idx] >> np.uint64(32)).astype(np.uint32),
                                r[idx] | np.uint32(t << 16), np.full(idx.size, bq, dtype=np.uint32), k0, k1)
            for qq in q[(q >> 3) == bq]:
                word = blk[(qq >> 1) & 3].astype(np.int64)
                draws[:, qq] = ((word >> 16) if qq & 1 else word) & 0x7FFF
        f = values[np.searchsorted(thr[: nv - 1], draws, side="right")]
        ok = (f.reshape(-1, 3, S) != 0).any(2).all(1)
        fac[idx[ok]] = f[ok]
        pending[idx[ok]] = False
    exhausted = int(pending.sum())
    unit = np.zeros(3 * S, dtype=np.int64)
    unit[[0, S, 2 * S]] = values[nv - 1]
    fac[pending] = unit
    tokens = (fac + shift).reshape(n, R, 3 * S).astype(np.int32)
    f3 = fac.reshape(n, R, 3, S)
    targets = np.einsum("nri,nrj,nrk->nijk", f3[:, :, 0], f3[:, :, 1], f3[:, :, 2]).astype(np.int32)
    return tokens, targets, exhausted


def demos_philox(seed: int, d0: int, n: int, values, probs, R: int, S: int, shift: int, max_tries: int = 64):
    """orc.demos_philox for any S: the C oracle where it holds the size, contract v1 restated above beyond."""
    if S <= 16:
        return orc.demos_philox(seed, d0, n, values, probs, R, S, shift, max_tries=max_tries)
    assert not orc.alias_applies(values, probs, S), "contract v2 is not defined beyond six groups per factor"
    return demos_philox_v1(seed, d0, n, values, probs, R, S, shift, max_tries)


# ---------------------------------------------------------------- parity mode (orc_demos_from_ustream)
def demos_from_ustream(ustream, values, probs, R: int, S: int, shift: int, n_demos: int):
    """The reference's rejection loop (utils.py:222-232) on a uniform stream: per try S doubles for u, S for v, S for w,
    value = first bucket whose float32 CDF >= u; rejected iff a factor is all zero.  -> (tokens, targets, consumed) for
    the complete demos."""
    u = np.asarray(ustream, dtype=np.float64)
    values = np.asarray(values, dtype=np.int64)
    cdf = orc.categorical_cdf(probs).astype(np.float64)
    ntry = len(u) // (3 * S)
    f = values[np.minimum(np.searchsorted(cdf, u[: ntry * 3 * S], side="left"), len(values) - 1)].reshape(ntry, 3, S)
    acc = np.nonzero((f != 0).any(2).all(1))[0]
    done = min(n_demos, len(acc) // R)
    take = acc[: done * R]
    fac = f[take].reshape(done, R, 3, S)
    tokens = (fac.reshape(done, R, 3 * S) + shift).astype(np.int32)
    targets = np.einsum("nri,nrj,nrk->nijk", fac[:, :, 0], fac[:, :, 1], fac[:, :, 2]).astype(np.int32)
    consumed = int(take[-1] + 1) * 3 * S if done else 0
    return tokens, targets, consumed


def demos_seeded(seed: int, values, probs, R: int, S: int, shift: int, n_demos: int, slack: float = 4.0):
    """Same as running the reference loop after torch.manual_seed(seed)."""
    probs32 = np.asarray(probs, dtype=np.float32)
    p0 = float(probs32[np.asarray(values) == 0].sum() / probs32.sum()) if 0 in list(values) else 0.0
    acc = max((1.0 - p0 ** S) ** 3, 1e-3)
    n_u = int(n_demos * R * 3 * S / acc * slack) + 4096
    while True:
        tok, tgt, used = demos_from_ustream(orc.mt_doubles(seed, n_u), values, probs, R, S, shift, n_demos)
        if len(tok) == n_demos:
            return tok, tgt, used
        n_u *= 2
