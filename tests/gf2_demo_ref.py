"""numpy restatement of tg_demo_gen_gf2 (include/tensorgame.h "mod-2 synthetic demonstrations") at any S: the alias tables
of contract v2 mod 2, built in the C oracle's operation order (orc_alias_build, orc_vose) so that the doubles match bit for
bit, the v2 draws, and contract v1 mod 2 on the Philox blocks of tests/oracle_any_s.py.  Test infrastructure only."""
from __future__ import annotations

import numpy as np

from oracle import tg_oracle as orc
from tests import oracle_any_s as oas

AB = 128  # buckets per table


def _norm(probs):
    total = 0.0
    for x in probs:
        total += float(x)
    return [float(x) / total for x in probs]


def p_even(values, probs) -> float:
    """P(value even) of the normalised alphabet, summed in the library's order."""
    p, pe = _norm(probs), 0.0
    for v, x in zip(values, p):
        if int(v) % 2 == 0:
            pe += x
    return pe


def alias_applies(values, probs, S: int) -> bool:
    """Contract v2 mod 2: at most five values, S <= 16, P(even) <= 0.999."""
    return 1 <= len(values) <= 5 and S in (4, 9, 16) and p_even(values, probs) <= 0.999


def vose(P, count: int) -> np.ndarray:
    """orc_vose: 128 buckets, 9-bit threshold | alias << 9."""
    sc = [(float(P[o]) if o < count else 0.0) * float(AB) for o in range(AB)]
    alias, prob = list(range(AB)), [1.0] * AB
    small = [o for o in range(AB) if sc[o] < 1.0]
    large = [o for o in range(AB) if not sc[o] < 1.0]
    while small and large:
        sm, lg = small.pop(), large.pop()
        prob[sm], alias[sm] = sc[sm], lg
        sc[lg] = (sc[lg] + sc[sm]) - 1.0
        (small if sc[lg] < 1.0 else large).append(lg)
    out = np.zeros(AB, dtype=np.uint16)
    for o in range(AB):
        q = min(max(prob[o], 0.0), 1.0)
        thr, al = int(q * 512.0 + 0.5), alias[o]
        if thr >= 512:
            thr, al = 511, o
        out[o] = thr | (al << 9)
    return out


def _outcome(o: int, size: int, n: int):
    """Value indices of outcome o of a group of `size` entries."""
    return [o % n, (o // n) % n, o // (n * n)] if size == 3 else [o]


def alias_tables(values, probs, S: int) -> np.ndarray:
    """uint16 (8, 128): [0] plain group of three, [1] plain single entry, [2 + g] tilted table of group g, where every
    all-even outcome is weighed by 1 - P(every later entry even)."""
    n, p, pe = len(values), _norm(probs), p_even(values, probs)
    ng = (S + 2) // 3
    last = S - 3 * (ng - 1)
    P3 = [(p[o % n] * p[(o // n) % n]) * p[o // (n * n)] for o in range(n ** 3)]
    tab = np.zeros((8, AB), dtype=np.uint16)
    tab[0], tab[1] = vose(P3, n ** 3), vose(p, n)
    for g in range(ng):
        size = 3 if g < ng - 1 else last
        count = n ** 3 if size == 3 else n
        qlater = 1.0
        for _ in range(3 * g + size, S):
            qlater *= pe
        W, s = [], 0.0
        for o in range(count):
            w = P3[o] if size == 3 else p[o]
            if all(int(values[i]) % 2 == 0 for i in _outcome(o, size, n)):
                w *= 1.0 - qlater
            W.append(w)
            s += w
        tab[2 + g] = vose([w / s for w in W], count)
    return tab


def _blocks(seed: int, d, r, t: int, nblk: int):
    k0, k1 = seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF
    lo, hi = (d & np.uint64(0xFFFFFFFF)).astype(np.uint32), (d >> np.uint64(32)).astype(np.uint32)
    c2 = (r.astype(np.uint32) | np.uint32(t << 16)).astype(np.uint32)
    return [oas.philox4x32_10(lo, hi, c2, np.full(len(d), b, dtype=np.uint32), k0, k1) for b in range(nblk)]


def _v2(seed, d, r, values, probs, S):
    """(pairs, 3, S) factor values under v2 mod 2."""
    vals, n = np.asarray(values, dtype=np.int64), len(values)
    tab = alias_tables(values, probs, S).astype(np.int64)
    ng = (S + 2) // 3
    last = S - 3 * (ng - 1)
    blk = _blocks(seed, d, r, 0, (3 * ng + 7) // 8)
    f = np.zeros((len(d), 3, S), dtype=np.int64)
    for fac in range(3):
        az = np.ones(len(d), dtype=bool)
        for g in range(ng):
            m = fac * ng + g
            word = blk[m >> 3][(m >> 1) & 3].astype(np.int64)
            h = (word >> 16) if m & 1 else word & 0xFFFF
            size = 3 if g < ng - 1 else last
            b = np.where(az, tab[2 + g][h & 127], tab[0 if size == 3 else 1][h & 127])
            o = np.where((h >> 7) < (b & 511), h & 127, b >> 9)
            e = vals[np.stack(_outcome(o, size, n), axis=1)]
            f[:, fac, 3 * g: 3 * g + size] = e
            az &= (e % 2 == 0).all(1)
    return f


def _v1(seed, d, r, values, probs, S, max_tries):
    """(pairs, 3, S) factor values and per-pair exhausted under v1 mod 2."""
    vals, nv = np.asarray(values, dtype=np.int64), len(values)
    thr = orc.philox_thresholds(probs).astype(np.int64)
    P = len(d)
    f = np.zeros((P, 3, S), dtype=np.int64)
    pending = np.ones(P, dtype=bool)
    for t in range(max_tries):
        idx = np.nonzero(pending)[0]
        if idx.size == 0:
            break
        blk = _blocks(seed, d[idx], r[idx], t, (3 * S + 7) // 8)
        draws = np.empty((idx.size, 3 * S), dtype=np.int64)
        for q in range(3 * S):
            word = blk[q >> 3][(q >> 1) & 3].astype(np.int64)
            draws[:, q] = ((word >> 16) if q & 1 else word) & 0x7FFF
        x = vals[np.searchsorted(thr[: nv - 1], draws, side="right")].reshape(-1, 3, S)
        ok = (x % 2 == 1).any(2).all(1)
        f[idx[ok]] = x[ok]
        pending[idx[ok]] = False
    odd = [int(v) for v in values if int(v) % 2]
    f[pending] = 0
    f[pending, :, 0] = odd[-1]
    return f, pending


def demos(seed: int, d0: int, n: int, values, probs, R: int, S: int, shift: int, max_tries: int = 64):
    """-> (tokens int32 (n, R, 3S), dense 0/1 targets uint8 (n, S, S, S), exhausted bool (n,)) of tg_demo_gen_gf2."""
    d = (np.uint64(d0) + np.repeat(np.arange(n, dtype=np.uint64), R)).astype(np.uint64)
    r = np.tile(np.arange(R, dtype=np.uint32), n)
    if alias_applies(values, probs, S):
        f, ex = _v2(seed, d, r, values, probs, S), np.zeros(n * R, dtype=bool)
    else:
        f, ex = _v1(seed, d, r, values, probs, S, max_tries)
    tokens = (f.reshape(n, R, 3 * S) + shift).astype(np.int32)
    b = (f & 1).reshape(n, R, 3, S)
    targets = (np.einsum("nri,nrj,nrk->nijk", b[:, :, 0], b[:, :, 1], b[:, :, 2]) & 1).astype(np.uint8)
    return tokens, targets, ex.reshape(n, R).any(1)
