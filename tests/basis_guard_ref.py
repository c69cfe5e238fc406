"""Model of the change of basis's path choice (tg_change_of_basis, tg_change_of_basis_i16), and the edge cases that pin it.

Every fast path of the change of basis is exact only inside a bound, and a guard per game decides which path computes
it; the exact int32 kernel (basis_kernel) redoes the games no guard accepts.  This module restates each guard in int64
numpy and Python integers, so that a test can say which path a game must take and which flag byte it must come back
with, and builds games on both sides of every threshold.

Notation (the kernels' contraction order: c with C, then b with B, then a with A):
    Y[a][b][k'] = sum_c C[k'][c] T[a][b][c]
    Z[a][j'][k'] = sum_b B[j'][b] Y[a][b][k']
    T'[i'][j'][k'] = sum_a A[i'][a] Z[a][j'][k']
n_M is the largest absolute row sum of M; tb = OR over the game of mag(x) + 1 with mag(x) = x for x >= 0 and -x-1
otherwise (an upper bound of max|T| that a warp forms with one OR reduction)."""
from dataclasses import dataclass

import numpy as np

from tests.test_edges_ref import change_of_basis_ref

RANGE, TOKEN_RANGE, PATH_PLANES, PATH_EXACT, REDO = 4, 16, 32, 64, 0x80

# f16 holds every integer up to 2048, and an operand that rounded is >= 2048 after rounding: the f16 operands (Y and Z)
# are accepted while their bound or their checked value is at most this
F16_OPERAND_MAX = 2047
# the 16-bit results of the f16 and byte-plane paths, the 9x9x9 int16 store without range test and the 16-bit packed
# lanes at 4x4x4 are exact while |value| is at most this
BITS16_MAX = 32767
# byte planes: ||C|| that keeps Y inside 16 bits
PLANES_NC_MAX = 255
# byte planes: ybound = PLANES_HI_SCALE * (OR of mag(high byte of Y) + 1)
PLANES_HI_SCALE = 256
# mats alignment (bytes, of the pointer and of the per-game stride) that routes 16x16x16 to the tensor cores and 4x4x4 to
# one thread per game
ALIGN_MMA16, ALIGN_THREAD4 = 4, 16
ZONE = {"int8": (-64, 63), "int16": (-32768, 32767)}


def mag(x) -> np.ndarray:
    x = np.asarray(x, dtype=np.int64)
    return np.where(x >= 0, x, -x - 1)


def or_bound(x) -> int:
    """OR over mag(x) + 1 (>= max|x|, inflated by the OR: {1, 2} -> 4)."""
    return int(np.bitwise_or.reduce(mag(x).ravel(), initial=0)) + 1


def norm(M) -> int:
    return int(np.abs(np.asarray(M, dtype=np.int64)).sum(axis=1).max())


def hi8(Y) -> np.ndarray:
    """The signed second byte of each value's low 16 bits (the high byte plane of the P16 path)."""
    w = np.asarray(Y, dtype=np.int64) & 0xFFFF
    h = w >> 8
    return np.where(h >= 128, h - 256, h)


def contract(T, A, B, C):
    """(Y, Z, T') in int64, in the kernels' order."""
    T, A, B, C = (np.asarray(x, dtype=np.int64) for x in (T, A, B, C))
    Y = np.einsum("kc,abc->abk", C, T)
    Z = np.einsum("jb,abk->ajk", B, Y)
    return Y, Z, np.einsum("ia,ajk->ijk", A, Z)


@dataclass
class Guard:
    ref: np.ndarray   # exact T'
    Y: np.ndarray
    Z: np.ndarray
    tb: int
    nA: int
    nB: int
    nC: int
    ybound: int       # P16's bound of max|Y| (from the high byte plane)
    path: str         # f16_apriori | f16_checked | planes | exact (16); f16_apriori | f16_tracked | exact (9);
                      # thread | lanes | exact (4)
    unchecked16: bool # int16 results are stored without a range test (P16, 9x9x9 without check3, 4x4x4 lanes)
    flags: int        # the flag byte the library must return


def model(T, A, B, C, out: str = "int8", align: int = 16) -> Guard:
    """The path and flag byte of one game.  out: 'int8' or 'int16'; align: the largest power of two (up to 16) that
    divides both the mats pointer and its per-game stride."""
    assert out in ZONE
    T = np.asarray(T, dtype=np.int64)
    S = T.shape[0]
    A, B, C = (np.asarray(x, dtype=np.int64) for x in (A, B, C))
    Y, Z, ref = contract(T, A, B, C)
    assert np.array_equal(ref, change_of_basis_ref(T, A, B, C))
    tb, nA, nB, nC = or_bound(T), norm(A), norm(B), norm(C)
    ybound = PLANES_HI_SCALE * (int(np.bitwise_or.reduce(mag(hi8(Y)).ravel(), initial=0)) + 1)
    ym, zm = int(np.abs(Y).max()), int(np.abs(Z).max())
    o16 = out == "int16"
    unchecked16 = False
    if S == 16:
        yb, zb = tb * nC, tb * nC * nB
        if align % ALIGN_MMA16:
            path = "exact"
        elif yb <= F16_OPERAND_MAX and zb <= F16_OPERAND_MAX and (o16 or zb * nA <= BITS16_MAX):
            path = "f16_apriori"
        elif ym <= F16_OPERAND_MAX and zm <= F16_OPERAND_MAX and (o16 or zm * nA <= BITS16_MAX):
            path = "f16_checked"
        elif nC <= PLANES_NC_MAX and ybound * nA * nB <= BITS16_MAX:
            path, unchecked16 = "planes", o16
        else:
            path = "exact"
    elif S == 9:
        if tb * nC <= F16_OPERAND_MAX and tb * nC * nB <= F16_OPERAND_MAX:
            path, unchecked16 = "f16_apriori", o16 and tb * nC * nB * nA <= BITS16_MAX
        elif ym <= F16_OPERAND_MAX and zm <= F16_OPERAND_MAX:
            path = "f16_tracked"
        else:
            path = "exact"
    elif S == 4:
        za = ym * nA
        if align % ALIGN_THREAD4 == 0:
            path = "thread"
        elif za <= BITS16_MAX and za * nB <= BITS16_MAX:
            path, unchecked16 = "lanes", o16
        else:
            path = "exact"
    else:
        raise ValueError(f"no change of basis at S = {S}")
    lo, hi = ZONE[out]
    flags = (RANGE if ((ref < lo) | (ref > hi)).any() else 0) | {"planes": PATH_PLANES, "exact": PATH_EXACT}.get(path, 0)
    return Guard(ref, Y, Z, tb, nA, nB, nC, ybound, path, unchecked16, flags)


# ---------------------------------------------------------------------------------------------------------------- cases
@dataclass
class Case:
    name: str
    T: np.ndarray
    A: np.ndarray
    B: np.ndarray
    C: np.ndarray
    out: str          # output the claims are about
    claims: dict      # model attribute or derived quantity -> value (checked by tests/test_basis_guards_ref.py)
    align: int = 16   # 4x4x4 cases that need the packed-lane kernel say 4

    @property
    def S(self) -> int:
        return self.T.shape[0]


def eye(S):
    return np.eye(S, dtype=np.int64)


def zeros(S, n=2):
    return np.zeros((S,) * n, dtype=np.int64)


def row(S, vals, r=0):
    """An S x S matrix whose row r is vals (zero-padded) and whose other rows are zero."""
    M = zeros(S)
    M[r, : len(vals)] = vals
    return M


def row_all(S, vals):
    """Every row of the S x S matrix is vals (zero-padded)."""
    M = zeros(S)
    M[:, : len(vals)] = vals
    return M


def sum_row(S, total):
    """A row of at most S non-negative int8 entries summing to total (as even as possible)."""
    q, r = divmod(total, S)
    assert q + (r > 0) <= 127
    return [q + (i < r) for i in range(S)]


def derived(g: Guard) -> dict:
    """Quantities the claims may name besides the model's fields."""
    ym, zm = int(np.abs(g.Y).max()), int(np.abs(g.Z).max())
    return {"maxY": ym, "maxZ": zm, "maxT'": int(np.abs(g.ref).max()), "yb": g.tb * g.nC, "zb": g.tb * g.nC * g.nB,
            "tb*nC*nB*nA": g.tb * g.nC * g.nB * g.nA, "maxZ*nA": zm * g.nA, "ybound*nA*nB": g.ybound * g.nA * g.nB,
            "maxY*nA*nB": ym * g.nA * g.nB, "T'[0,0,0]": int(g.ref[0, 0, 0])}


def cases16() -> list[Case]:
    S, out = 16, []
    I = eye(S)
    T23 = np.full((S,) * 3, -23, dtype=np.int64)
    T128 = np.full((S,) * 3, -128, dtype=np.int64)
    for sg in (1, -1):  # sg flips the sign of Y (and of everything after it)
        # a-priori yb = tb nC: -23 * 89 = -2047 (f16 without checks) vs -128 * 16 = -2048
        out.append(Case(f"16 yb=2047 sg{sg}", T23, I, I, sg * row(S, sum_row(S, 89)), "int8",
                        {"tb": 23, "nC": 89, "yb": 2047, "maxY": 2047, "path": "f16_apriori"}))
        out.append(Case(f"16 yb=2048 sg{sg}", T128, I, I, sg * row(S, [1] * 16), "int8",
                        {"tb": 128, "yb": 2048, "maxY": 2048, "path": "planes"}))
        # the same with B = 0 (zb = 0): only the yb test keeps Y = 2048 off the unchecked path
        out.append(Case(f"16 yb=2048 zb=0 sg{sg}", T128, I, zeros(S), sg * row(S, [1] * 16), "int8",
                        {"yb": 2048, "zb": 0, "maxY": 2048, "path": "planes"}))
        # a-priori zb = tb nC nB: -23 * 1 * 89 vs -128 * 1 * 16
        out.append(Case(f"16 zb=2047 sg{sg}", T23, I, sg * row(S, sum_row(S, 89)), I, "int8",
                        {"yb": 23, "zb": 2047, "maxZ": 2047, "path": "f16_apriori"}))
        out.append(Case(f"16 zb=2048 sg{sg}", T128, I, sg * row(S, [1] * 16), I, "int8",
                        {"yb": 128, "zb": 2048, "maxZ": 2048, "ybound": 256, "path": "planes"}))
        # checked |Y| = 2047 / 2048 / 2049 (T entries -128 and +-1 at c = 0, 1 of b = 0; B = 0 so that Z stays 0)
        for y, t1, c in ((2047, 1, [16, 1]), (2048, 0, [16]), (2049, -1, [-16, -1])):
            T = zeros(S, 3)
            T[:, 0, 0], T[:, 0, 1] = -128, t1
            out.append(Case(f"16 checked Y={y} sg{sg}", T, I, zeros(S), sg * row(S, c), "int8",
                            {"maxY": y, "maxZ": 0, "path": "f16_checked" if y == 2047 else "planes"}))
        # checked |Z| = 2047 / 2048 / 2049 (C = I so Y = T; B row 0 picks T[a][0][0] = -128 and T[a][1][0])
        for z, t1, b in ((2047, -127, [15, 1]), (2048, 0, [16]), (2049, -1, [-16, -1])):
            T = zeros(S, 3)
            T[:, 0, 0], T[:, 1, 0] = -128, t1
            out.append(Case(f"16 checked Z={z} sg{sg}", T, I, sg * row(S, b), I, "int8",
                            {"maxY": 128, "maxZ": z, "zb": 128 * sum(map(abs, b)),
                             "path": "f16_checked" if z == 2047 else "planes"}))
        # the OR-inflated tb: entries {64, 63} give tb = 128 (max|T| = 64): the a-priori bound fails, the checked path holds
        T = zeros(S, 3)
        T[:, :, 0], T[:, :, 1] = 64, 63
        out.append(Case(f"16 tb inflated sg{sg}", T, I, I, sg * row(S, [16]), "int8",
                        {"tb": 128, "yb": 2048, "maxY": 1024, "path": "f16_checked"}))
        out.append(Case(f"16 tb tight sg{sg}", np.full((S,) * 3, 64, dtype=np.int64), I, I, sg * row(S, [16]), "int8",
                        {"tb": 65, "yb": 1040, "maxY": 1024, "path": "f16_apriori"}))
    # int8 out: max|Z| nA = 2047 * 16 = 32752 (f16) vs 2047 * 17 = 34799 (the low 16 bits would not hold T')
    Tz = zeros(S, 3)
    Tz[:, 0, 0], Tz[:, 1, 0] = -128, -127
    for sg in (1, -1):
        for arow, prod, path in (([1] * 16, 32752, "f16_checked"), ([2] + [1] * 15, 34799, "exact")):
            out.append(Case(f"16 maxZ*nA={prod} sg{sg}", Tz, sg * row_all(S, arow), row(S, [15, 1]), I, "int8",
                            {"maxZ": 2047, "maxZ*nA": prod, "path": path, "T'[0,0,0]": -sg * prod}))
            out.append(Case(f"16 maxZ*nA={prod} int16 sg{sg}", Tz, sg * row_all(S, arow), row(S, [15, 1]), I, "int16",
                            {"maxZ": 2047, "path": "f16_checked", "flags": RANGE if prod > BITS16_MAX else 0}))
    # the alias: Z = 2047 for every a, an A row summing to 32: T' = 65504 = -32 mod 2^16 (in the int8 zone)
    out.append(Case("16 alias 65504", Tz, row(S, [2] * 16), -row(S, [15, 1]), I, "int8",
                    {"maxZ": 2047, "maxZ*nA": 65504, "T'[0,0,0]": 65504, "path": "exact", "flags": RANGE | PATH_EXACT}))
    # P16: ybound nA nB = 256 * 1 * 127 = 32512 (planes) vs 256 * 16 * 8 = 32768 (exact); Y = -256 from C rows (1, 1)
    C11 = row_all(S, [1, 1])
    for sg in (1, -1):
        out.append(Case(f"16 planes 32512 sg{sg}", T128, sg * I, row_all(S, [127]), C11, "int16",
                        {"maxY": 256, "ybound": 256, "nC": 2, "ybound*nA*nB": 32512, "T'[0,0,0]": -sg * 32512,
                         "path": "planes", "flags": PATH_PLANES}))
        out.append(Case(f"16 planes 32768 sg{sg}", T128, sg * row_all(S, [1] * 16), row_all(S, [1] * 8), C11, "int16",
                        {"maxY": 256, "maxZ": 2048, "ybound*nA*nB": 32768, "T'[0,0,0]": -sg * 32768, "path": "exact",
                         "flags": PATH_EXACT | (RANGE if sg < 0 else 0)}))
    # nC = 255 (planes) vs 256 (exact): one entry -128, Y = -16256 (high byte -64: ybound = 16384)
    T1 = zeros(S, 3)
    T1[0, 0, 0] = -128
    for sg in (1, -1):
        for c, path in (([127, 127, 1], "planes"), ([127, 127, 2], "exact")):
            out.append(Case(f"16 nC={sum(c)} sg{sg}", T1, I, I, sg * row(S, c), "int16",
                            {"nC": sum(c), "maxY": 16256, "ybound": 16384, "path": path}))
    # Y = 4 * 128 * 128 = 65536 is 0 in 16 bits (ybound 256): only the nC test keeps it off the byte planes
    T4 = zeros(S, 3)
    T4[0, 0, :4] = -128
    out.append(Case("16 Y=65536 wraps to 0", T4, I, I, row(S, [-128] * 4), "int16",
                    {"nC": 512, "maxY": 65536, "ybound": 256, "path": "exact", "flags": RANGE | PATH_EXACT}))
    return out


def cases9() -> list[Case]:
    S, out = 9, []
    I = eye(S)
    T23 = np.full((S,) * 3, -23, dtype=np.int64)
    T128 = np.full((S,) * 3, -128, dtype=np.int64)
    for sg in (1, -1):
        # a-priori tb nc and tb nc nb = 2047 (f16 accumulators) vs 2048
        out.append(Case(f"9 tb*nc=2047 sg{sg}", T23, I, I, sg * row(S, sum_row(S, 89)), "int8",
                        {"yb": 2047, "maxY": 2047, "path": "f16_apriori"}))
        out.append(Case(f"9 tb*nc=2048 sg{sg}", T128, I, I, sg * row(S, [2] * 8), "int8",
                        {"yb": 2048, "maxY": 2048, "path": "exact"}))
        out.append(Case(f"9 tb*nc*nb=2047 sg{sg}", T23, I, sg * row(S, sum_row(S, 89)), I, "int8",
                        {"yb": 23, "zb": 2047, "maxZ": 2047, "path": "f16_apriori"}))
        out.append(Case(f"9 tb*nc*nb=2048 sg{sg}", T128, I, sg * row(S, [2] * 8), I, "int8",
                        {"zb": 2048, "maxZ": 2048, "path": "exact"}))
        # tracked |Y| = 2047 / 2048 / 2049 (B = I: Z = Y)
        for y, t1, c in ((2047, 1, [16, 1]), (2048, 0, [16]), (2049, -1, [-16, -1])):
            T = zeros(S, 3)
            T[:, 0, 0], T[:, 0, 1] = -128, t1
            out.append(Case(f"9 tracked Y={y} sg{sg}", T, I, I, sg * row(S, c), "int8",
                            {"maxY": y, "path": "f16_tracked" if y == 2047 else "exact"}))
        # tracked |Z| = 2047 / 2048 / 2049 (C = I: Y = T)
        for z, t1, b in ((2047, -127, [15, 1]), (2048, 0, [16]), (2049, -1, [-16, -1])):
            T = zeros(S, 3)
            T[:, 0, 0], T[:, 1, 0] = -128, t1
            out.append(Case(f"9 tracked Z={z} sg{sg}", T, I, sg * row(S, b), I, "int8",
                            {"maxY": 128, "maxZ": z, "path": "f16_tracked" if z == 2047 else "exact"}))
        # int16 out without range test while tb nc nb na <= 32767: na = 255 (T' = +-32640) vs na = 256 (T' = -32768 fits,
        # +32768 does not)
        for arow, t in (([-128, -127], 32640), ([127, 127, 1], -32640), ([127, 127, 2], -32768), ([-128, -128], 32768)):
            out.append(Case(f"9 int16 T'={t} sg{sg}", T128, row(S, arow), sg * I, I, "int16",
                            {"tb*nC*nB*nA": 128 * sum(map(abs, arow)), "T'[0,0,0]": sg * t,
                             "unchecked16": 128 * sum(map(abs, arow)) <= BITS16_MAX,
                             "flags": RANGE if sg * t > BITS16_MAX else 0}))
        # the largest |T'| the f16 path allows: Z = 2047 at every a, an A row of nine -128 (1152)
        out.append(Case(f"9 T'=2047*1152 sg{sg}", T23, row(S, [-128] * 9), I, sg * row(S, sum_row(S, 89)), "int8",
                        {"maxZ": 2047, "nA": 1152, "T'[0,0,0]": sg * 2047 * 1152, "path": "f16_apriori"}))
    # int8 out at the zone's edges, from two entries through C row (1, 1)
    for v in (-65, -64, 63, 64):
        T = zeros(S, 3)
        T[0, 0, 0], T[0, 0, 1] = v // 2, v - v // 2
        out.append(Case(f"9 int8 T'={v}", T, I, I, row(S, [1, 1]), "int8",
                        {"T'[0,0,0]": v, "path": "f16_apriori", "flags": RANGE if v in (-65, 64) else 0}))
    return out


def cases4() -> list[Case]:
    """Mats not 16-byte aligned: the packed-lane kernel (16-bit lanes), guard max|Y| nA <= 32767 and max|Y| nA nB <= 32767."""
    S, out = 4, []
    C11 = row_all(S, [1, 1])
    T151 = zeros(S, 3)
    T151[:, :, 0], T151[:, :, 1] = -128, -23  # Y = -151 everywhere
    T128 = np.full((S,) * 3, -128, dtype=np.int64)
    for sg in (1, -1):
        # 151 * 7 * 31 = 32767: T' = -+32767 on the lanes
        out.append(Case(f"4 lanes 32767 sg{sg}", T151, sg * row_all(S, [4, 3]), row_all(S, [8, 8, 8, 7]), C11, "int16",
                        {"maxY": 151, "maxY*nA*nB": 32767, "T'[0,0,0]": -sg * 32767, "path": "lanes", "flags": 0},
                        align=4))
        # 128 * 16 * 16 = 32768: T' = -+32768, redone exactly (+32768 does not fit int16)
        out.append(Case(f"4 lanes 32768 sg{sg}", T128, sg * row_all(S, [4] * 4), row_all(S, [4] * 4), eye(S), "int16",
                        {"maxY": 128, "maxY*nA*nB": 32768, "T'[0,0,0]": -sg * 32768, "path": "exact",
                         "flags": PATH_EXACT | (RANGE if sg < 0 else 0)}, align=4))
    return out


def all_cases() -> list[Case]:
    return cases16() + cases9() + cases4()
