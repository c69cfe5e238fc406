"""Numpy restatement of contract box v1 (tg_demo_gen_box, tg_demo_gen_box_gf2) and of the rectangular matmul tensors.

Box v1 is contract v1 at size S (oracle_any_s.demos_philox_v1) with the factors confined to the box (nu, nv, nw): every
try draws all 3S values as v1 does, the entries outside the box become 0, and a try is accepted iff u, v and w each have
a non-zero (mod 2: an odd) entry inside the box.  After max_tries the term is u = v = w = x e_0, x the last value (mod 2
the last odd value), and the demo is EXHAUSTED.
"""
from __future__ import annotations

import itertools

import numpy as np

from oracle import tg_oracle as orc
from tests import oracle_any_s as oas

SIZES = (4, 9, 16, 25)


def matmul_box(n: int, m: int, p: int):
    box = (n * m, m * p, n * p)
    return next(S for S in SIZES if max(box) <= S), box


def matmul_tensor(n: int, m: int, p: int, S: int) -> np.ndarray:
    """T[i m + j][j p + k][i p + k] = 1, zero-padded to (S, S, S)."""
    T = np.zeros((S, S, S), dtype=np.int64)
    for i, j, k in itertools.product(range(n), range(m), range(p)):
        T[i * m + j, j * p + k, i * p + k] = 1
    return T


def naive_factors(n: int, m: int, p: int, S: int) -> np.ndarray:
    """The n m p terms e_{i m + j} (x) e_{j p + k} (x) e_{i p + k}: (n m p, 3, S) coefficients."""
    out = np.zeros((n * m * p, 3, S), dtype=np.int64)
    for t, (i, j, k) in enumerate(itertools.product(range(n), range(m), range(p))):
        out[t, 0, i * m + j] = out[t, 1, j * p + k] = out[t, 2, i * p + k] = 1
    return out


def shapes():
    """Every <n, m, p> with n, m, p <= 5, as (n, m, p, S, box)."""
    return [(n, m, p) + matmul_box(n, m, p) for n, m, p in itertools.product(range(1, 6), repeat=3)]


def inside(S: int, box) -> np.ndarray:
    """(3, S) bool: entry e of factor f lies in the box."""
    return np.arange(S)[None, :] < np.asarray(box)[:, None]


def demos(seed: int, d0: int, n: int, values, probs, R: int, S: int, shift: int, box, max_tries: int = 64, gf2: bool = False):
    """-> (tokens int32 (n, R, 3S), targets (n, S, S, S) -- integer, or 0/1 uint8 mod 2 --, exhausted bool (n,))."""
    vals = np.asarray(values, dtype=np.int64)
    thr = orc.philox_thresholds(probs).astype(np.int64)
    nv = len(vals)
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    d = (np.uint64(d0) + np.repeat(np.arange(n, dtype=np.uint64), R)).astype(np.uint64)
    r = np.tile(np.arange(R, dtype=np.uint32), n)
    P = n * R
    ins = inside(S, box)
    fac = np.zeros((P, 3, S), dtype=np.int64)
    pending = np.ones(P, dtype=bool)
    for t in range(max_tries):
        idx = np.nonzero(pending)[0]
        if idx.size == 0:
            break
        draws = np.empty((idx.size, 3 * S), dtype=np.int64)
        for bq in range((3 * S + 7) // 8):
            blk = oas.philox4x32_10((d[idx] & np.uint64(0xFFFFFFFF)).astype(np.uint32), (d[idx] >> np.uint64(32)).astype(np.uint32),
                                    r[idx] | np.uint32(t << 16), np.full(idx.size, bq, dtype=np.uint32), k0, k1)
            for q in range(8 * bq, min(8 * bq + 8, 3 * S)):
                word = blk[(q >> 1) & 3].astype(np.int64)
                draws[:, q] = ((word >> 16) if q & 1 else word) & 0x7FFF
        f = vals[np.searchsorted(thr[: nv - 1], draws, side="right")].reshape(-1, 3, S) * ins
        ok = ((f % 2 == 1) if gf2 else (f != 0)).any(2).all(1)
        fac[idx[ok]] = f[ok]
        pending[idx[ok]] = False
    x = [int(v) for v in values if int(v) % 2][-1] if gf2 else int(vals[-1])
    fac[pending] = 0
    fac[pending, :, 0] = x
    tokens = (fac.reshape(n, R, 3 * S) + shift).astype(np.int32)
    f3 = fac.reshape(n, R, 3, S)
    if gf2:
        b = f3 & 1
        targets = (np.einsum("nri,nrj,nrk->nijk", b[:, :, 0], b[:, :, 1], b[:, :, 2]) & 1).astype(np.uint8)
    else:
        targets = np.einsum("nri,nrj,nrk->nijk", f3[:, :, 0], f3[:, :, 1], f3[:, :, 2])
    return tokens, targets, pending.reshape(n, R).any(1)


def range_flags(targets) -> np.ndarray:
    """TG_FLAG_RANGE of the integer targets: an entry outside [-64, 63]."""
    t = np.asarray(targets)
    return ((t < -64) | (t > 63)).reshape(len(t), -1).any(1)


def box_bases(mats, box) -> np.ndarray:
    """env.box_bases on integer triples (N, 3, S, S): leading box[f] x box[f] block of matrix f, identity elsewhere."""
    m = np.array(mats, dtype=np.int64, copy=True)
    S = m.shape[-1]
    for f, k in enumerate(box):
        blk = np.eye(S, dtype=np.int64)
        blk = np.broadcast_to(blk, m[:, f].shape).copy()
        blk[:, :k, :k] = m[:, f, :k, :k]
        m[:, f] = blk
    return m
