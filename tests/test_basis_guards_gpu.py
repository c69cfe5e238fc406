"""The change of basis's fast-path guards at their thresholds, path by path, on the GPU.

Every case of tests/basis_guard_ref.py runs through both entry points (int8 and int16 out), with one triple per game and
with one shared triple, mixed with identity and random games so that every warp and CTA holds more than one kind of
game, and with the matrices at several byte offsets (which route 4x4x4 and 16x16x16 to different kernels).  The flag
byte must equal the model's bit for bit: RANGE, PATH_PLANES and PATH_EXACT say which guard held; a guard that is off by
one moves a game to another path (a different flag byte) or lets a fast path store a wrong value without RANGE.
Also here: the exact kernel's redo scheduler beyond one window of 1024 games per CTA, tg_change_of_basis_factors at
the token edges, and tg_sample_unimodular against the oracle."""
import numpy as np
import pytest
import torch

from oracle import tg_oracle as orc
from tests import basis_guard_ref as gr
from tests.helpers import dense_to_slab, geo, tape3_to_tokens, tokens_to_tape3
from tests.test_edges_ref import det_int

pytestmark = pytest.mark.gpu

DTYPES = {"int8": torch.int8, "int16": torch.int16}


@pytest.fixture(scope="module")
def env():
    from mat_mul_b200 import env as e

    assert torch.cuda.is_available()
    return e


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def place(m: np.ndarray, off: int) -> torch.Tensor:
    """int8 copy of m on the device whose first byte sits `off` bytes past a 16-byte boundary (off = 0: 16-aligned)."""
    buf = torch.zeros(m.size + 64, dtype=torch.int8, device="cuda")
    base = (-buf.data_ptr()) % 16 + off
    view = buf[base:base + m.size].view(m.shape)
    view.copy_(torch.from_numpy(m.astype(np.int8)))
    assert view.data_ptr() % 16 == off
    return view


def dense(out: torch.Tensor, S: int) -> np.ndarray:
    """int8 or int16 slab -> (N,S,S,S) int64, padding ignored."""
    rp, _, _ = geo(S)
    return out.cpu().numpy()[:, : S * rp].reshape(-1, S, rp)[:, :, : S * S].reshape(-1, S, S, S).astype(np.int64)


def check(out, flags, models, S, out_name, tag=""):
    """The flag byte of every game equals the model's; int16 out equals T' where it fits; int8 out equals T' inside the
    zone and its low byte everywhere."""
    f = flags.cpu().numpy()
    want_f = np.array([g.flags for g in models], dtype=np.uint8)
    bad = np.nonzero(f != want_f)[0]
    assert len(bad) == 0, [(int(n), models[n].path, hex(f[n]), hex(want_f[n]), tag) for n in bad[:8]]
    got, ref = dense(out, S), np.stack([g.ref for g in models])
    fits = (want_f & gr.RANGE) == 0
    wrong = np.nonzero(~(got == ref).reshape(len(ref), -1).all(1) & fits)[0]
    assert len(wrong) == 0, [(int(n), models[n].path, tag) for n in wrong[:8]]
    if out_name == "int8":
        assert np.array_equal(got & 0xFF, ref & 0xFF), tag


def fillers(S, n, rng):
    """n filler games with their triples: identity matrices on full-range games, and small sparse matrices."""
    out = []
    for q in range(n):
        T = rng.integers(-128, 128, (S, S, S)) * (rng.random((S, S, S)) < 0.5)
        if q % 2 == 0:
            m = np.stack([np.eye(S, dtype=np.int64)] * 3)
        else:
            T = np.clip(T, -4, 4)
            m = np.eye(S, dtype=np.int64) + rng.integers(-1, 2, (3, S, S)) * (rng.random((3, S, S)) < 0.1)
        out.append((T, m))
    return out


def cases_of(S):
    return [c for c in gr.all_cases() if c.S == S]


OFFSETS = [(16, 0), (16, 1), (16, 2), (16, 3), (16, 4), (16, 8), (9, 0), (9, 1), (9, 2), (9, 3), (9, 4), (9, 8),
           (4, 0), (4, 4), (4, 8)]


@pytest.mark.parametrize("S,off", OFFSETS)
@pytest.mark.parametrize("out_name", ["int8", "int16"])
def test_guard_cases_one_triple_per_game(env, S, off, out_name):
    """Each case between two fillers; the mats at byte offset `off` (16x16x16: any offset not a multiple of 4 sends every
    game to the exact kernel; 4x4x4: any offset not a multiple of 16 sends it to the packed lanes)."""
    rng = np.random.default_rng(1000 * S + off)
    games = []
    for c in cases_of(S):
        f0, f1 = fillers(S, 2, rng)
        games += [f0, (c.T, np.stack([c.A, c.B, c.C])), f1]
    T = np.stack([g[0] for g in games])
    m = np.stack([g[1] for g in games])
    align = off or 16
    models = [gr.model(t, *mm, out_name, align) for t, mm in zip(T, m)]
    if S == 16 and align % 4:
        assert all(g.path == "exact" for g in models)
    out, flags = env.change_of_basis(dev(dense_to_slab(T)), place(m, off), S, out_dtype=DTYPES[out_name])
    check(out, flags, models, S, out_name, f"S={S} off={off}")


@pytest.mark.parametrize("S,off", [(16, 0), (9, 0), (9, 3), (4, 0), (4, 4)])
@pytest.mark.parametrize("out_name", ["int8", "int16"])
def test_guard_cases_shared_triple(env, S, off, out_name):
    """Each case's triple shared by its own game and by fillers of other kinds (identity-like and full-range games)."""
    rng = np.random.default_rng(2000 * S + off)
    align = off or 16
    for c in cases_of(S):
        T = [rng.integers(-3, 4, (S, S, S)), c.T, rng.integers(-128, 128, (S, S, S)), np.zeros((S, S, S), np.int64), c.T[::-1]]
        T = np.stack(T + [t[:, ::-1] for t in T])
        m = np.stack([c.A, c.B, c.C])[None]
        models = [gr.model(t, c.A, c.B, c.C, out_name, align) for t in T]
        out, flags = env.change_of_basis(dev(dense_to_slab(T)), place(m, off), S, out_dtype=DTYPES[out_name])
        check(out, flags, models, S, out_name, c.name)


def test_redo_scheduler_beyond_one_window(env):
    """basis_kernel's redo pass gives each of at most 148 * 32 CTAs a contiguous chunk of the flags and walks it in windows
    of 1024 games.  With N = 4 853 000 a chunk is 1025 games, so the second window of a chunk holds one game, and the
    last chunk is partial (650 games).  Games marked by the packed-lane kernel (4x4x4, mats at offset 4) sit at chunk
    offsets 0, 1023 and 1024 of the first, a middle and the last full CTA, and at both ends of the partial chunk."""
    S, N, grid = 4, 4_853_000, 148 * 32
    chunk = -(-N // grid)
    assert chunk == 1025 and N - (N // chunk) * chunk == 650
    marked = []
    for cta in (0, 2000, N // chunk - 1):
        marked += [cta * chunk + o for o in (0, 1023, 1024)]
    last = (N // chunk) * chunk
    marked += [last, last + 1, N - 1]
    assert max(marked) == N - 1 and len(set(marked)) == len(marked)
    cases = [c for c in cases_of(4) if c.claims.get("path") == "exact"]  # max|Y| nA nB = 32768: T' = -32768 or +32768
    assert len(cases) == 2
    gen = torch.Generator(device="cuda").manual_seed(7)
    slab = torch.randint(-128, 128, (N, 64), dtype=torch.int8, device="cuda", generator=gen)
    buf = torch.empty(N * 48 + 64, dtype=torch.int8, device="cuda")
    base = (-buf.data_ptr()) % 16 + 4
    mats = buf[base:base + N * 48].view(N, 3, S, S)
    mats.copy_(torch.eye(S, dtype=torch.int8, device="cuda").expand(N, 3, S, S))
    models = {}
    for q, n in enumerate(marked):
        c = cases[q % 2]
        slab[n] = dev(dense_to_slab(c.T[None]))[0]
        mats[n] = dev(np.stack([c.A, c.B, c.C]).astype(np.int8))
        models[n] = gr.model(c.T, c.A, c.B, c.C, "int16", align=4)
        assert models[n].path == "exact"
    out, flags = env.change_of_basis(slab, mats, S, out_dtype=torch.int16)
    idx = torch.tensor(marked, device="cuda")
    fm = flags[idx].cpu().numpy()
    assert list(fm) == [models[n].flags for n in marked]
    got = dense(out[idx], S)
    for q, n in enumerate(marked):
        if not models[n].flags & gr.RANGE:
            assert np.array_equal(got[q], models[n].ref), n
    # every other game: identity matrices, so T' = T on the fast path, unflagged
    keep = torch.ones(N, dtype=torch.bool, device="cuda")
    keep[idx] = False
    assert int(flags[keep].count_nonzero()) == 0
    assert torch.equal(out[keep], slab[keep].to(torch.int16))


# ---------------------------------------------------------------- tg_change_of_basis_factors
def edge_factors(S, R, N, shift_in, rng):
    """Coefficients (N,R,3,S) in [-shift_in, 255 - shift_in] and per-game matrices I + e_0 e_1^T with row 1 negated:
    coef'_0 = u_0 + u_1 and coef'_1 = -u_1.  Pairs (u_0, u_1) put coef'_0 on +-127, +-128 (shift_out = 127: the
    edge and one past) wherever the token range reaches them; the other coefficients stay inside +-60, so that every
    transformed one stays inside +-120."""
    lo, hi = -shift_in, 255 - shift_in
    fac = rng.integers(max(lo, -60), 61, (N, R, 3, S))
    targets = [t for t in (127, 128, -127, -128, 126, -126) if lo * 2 <= t <= hi * 2]
    for n in range(N):
        if n % 3 == 2:
            continue  # some games keep every coefficient inside
        t = targets[n % len(targets)]
        u0 = min(max(t, lo), hi)
        fac[n, n % R, n % 3, 0], fac[n, n % R, n % 3, 1] = u0, t - u0
    fac[1, 0, 2, 1] = hi  # a token of 255
    M = np.eye(S, dtype=np.int64)
    M[0, 1], M[1, 1] = 1, -1
    return fac, M


@pytest.mark.parametrize("S", [4, 9, 16])
@pytest.mark.parametrize("shift_in", [1, 64, 127])
@pytest.mark.parametrize("per_game", [True, False])
def test_factors_at_the_token_edges(env, S, shift_in, per_game):
    R, N, shift_out = 5, 48, 127
    rng = np.random.default_rng(S * 1000 + shift_in)
    fac, M = edge_factors(S, R, N, shift_in, rng)
    tok = (fac + shift_in).reshape(N, R, 3 * S)
    assert tok.min() >= 0 and tok.max() <= 255
    mats = np.stack([M, M.T.copy(), M])  # A, B, C
    m = np.stack([mats] * N) if per_game else mats[None]
    want = np.stack([orc.change_of_basis_factors(fac[n], *mats) for n in range(N)])  # (N,R,3,S)
    hit = np.abs(want).max(axis=(1, 2, 3))
    slab = dev(np.zeros((N, geo(S)[1]), dtype=np.int8))
    _, tape2, flags = env.change_of_basis(slab, dev(m.astype(np.int8)) if per_game else dev(mats.astype(np.int8)), S,
                                          tape=dev(tokens_to_tape3(tok)), shift=shift_in, shift_out=shift_out)
    f = flags.cpu().numpy()
    assert np.array_equal((f & gr.TOKEN_RANGE) != 0, hit > shift_out)
    got = tape3_to_tokens(tape2.cpu().numpy(), S).reshape(N, R, 3, S).astype(np.int64)
    assert np.array_equal(got, (want + shift_out) & 0xFF)
    if shift_in >= 64:  # both sides of the edge are reached
        assert (hit == 127).any() and (hit == 128).any()


@pytest.mark.parametrize("per_game", [True, False])
def test_factors_16_generic_kernel_equals_the_16_kernel(env, per_game):
    """tape_out at an odd address sends S = 16 to the generic basis_factors_kernel<16>; it must write the same bytes and
    flags as basis_factors16_kernel."""
    from mat_mul_b200 import _lib
    from mat_mul_b200.env import _p, _stream, check as check_rc, layout

    S, R, N, shift_in, shift_out = 16, 7, 101, 2, 100
    TP = layout(S).token_pitch
    rng = np.random.default_rng(16)
    tok = rng.integers(0, 2 * shift_in + 1, (N, R, 3 * S))
    tok[::7] = rng.integers(0, 256, (len(tok[::7]), R, 3 * S))  # over-bound tokens and large coefficients too
    m = rng.integers(-2, 3, (N if per_game else 1, 3, S, S)) * (rng.random((N if per_game else 1, 3, S, S)) < 0.3)
    m[0] = np.eye(S)
    tape = dev(tokens_to_tape3(tok))
    mats = dev(m.astype(np.int8))
    slab = dev(np.zeros((N, geo(S)[1]), dtype=np.int8))
    _, ref_tape, ref_flags = env.change_of_basis(slab, mats, S, tape=tape, shift=shift_in, shift_out=shift_out)
    buf = torch.full((R * N * TP + 32,), 0x5A, dtype=torch.uint8, device="cuda")
    base = (-buf.data_ptr()) % 16 + 1
    tape_out = buf[base:base + R * N * TP]
    flags = torch.zeros(N, dtype=torch.uint8, device="cuda")
    check_rc(_lib.lib().tg_change_of_basis_factors(_p(tape), N * TP, shift_in, _p(mats), int(per_game), _p(tape_out),
                                                   N * TP, shift_out, _p(flags), N, R, S, _stream()),
             "tg_change_of_basis_factors")
    assert torch.equal(tape_out, ref_tape.reshape(-1))
    assert torch.equal(flags, ref_flags & gr.TOKEN_RANGE)
    assert (buf[:base] == 0x5A).all() and (buf[base + R * N * TP:] == 0x5A).all()  # nothing outside the tape
    fac2 = tape3_to_tokens(ref_tape.cpu().numpy(), S).reshape(N, R, 3, S).astype(np.int64)
    fac = tok.reshape(N, R, 3, S) - shift_in
    for n in (0, 7, N - 1):
        want = orc.change_of_basis_factors(fac[n], *m[n if per_game else 0])
        assert np.array_equal(fac2[n], (want + shift_out) & 0xFF), n


# ---------------------------------------------------------------- tg_sample_unimodular
@pytest.mark.parametrize("S", [4, 9, 16])
@pytest.mark.parametrize("p", [0.0, 1 / 128 - 1e-9, 1 / 128, 0.5, 127 / 128, 1.0])
def test_sample_unimodular_against_the_oracle(env, S, p):
    N = 24
    got = env.sample_unimodular(N, S, seed=11, first=3, p_nonzero=p).cpu().numpy().astype(np.int64)
    assert np.array_equal(got, orc.sample_unimodular(11, 3, N, S, p))
    for M in got.reshape(-1, S, S):
        assert abs(det_int(M)) == 1
    off = (got.reshape(-1, S, S) * (1 - np.eye(S, dtype=np.int64))) != 0
    if int(p * 128) == 0:
        assert not off.any()  # below 1/128 the quantised probability is 0: diagonal matrices of +-1
    if p == 1.0:  # every off-diagonal entry of L and U is non-zero: the densest and largest matrices
        assert off.mean() > 0.6 and np.abs(got).max() >= 4
