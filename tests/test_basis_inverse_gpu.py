"""The inverse triples on a B200: tg_invert_bases (over Z at 4, 9 and 16) and tg_invert_bases_gf2 (over GF(2) at 4, 9, 16
and 25) bit for bit against tests/basis_inverse_ref.py, and end to end: a change of basis followed by its inverse returns
the demos mod 2, and factors moved into a random basis over Z map back to the original tape and target."""
import numpy as np
import pytest
import torch

from mat_mul_b200 import _lib, env
from tests import basis_inverse_ref as ref
from tests import gf2_basis_ref, i16_ref
from tests.helpers import slab_to_dense

pytestmark = pytest.mark.gpu

INT_SIZES = (4, 9, 16)
GF2_SIZES = (4, 9, 16, 25)
BATCHES = (1, 3, 257, 3000)
PROBS = (0.0, 1 / 128, 0.1, 0.3, 1.0)
FIRST = (1 << 32) - 2  # the Philox key changes within the batch
DEV = "cuda"


def _check_int(mats_np, inv, flags):
    want_inv, want_flags = ref.inverses_int8(mats_np)
    assert np.array_equal(flags.cpu().numpy(), want_flags)
    assert np.array_equal(inv.cpu().numpy().astype(np.int64), want_inv)
    return want_flags


@pytest.mark.parametrize("S", INT_SIZES)
@pytest.mark.parametrize("p", PROBS)
def test_sampled_unimodular_triples(S, p):
    for B in BATCHES:
        mats = env.sample_unimodular(B, S, seed=S, first=FIRST, p_nonzero=p)
        inv, flags = env.invert_bases(mats)
        assert inv.shape == (B, 3, S, S) and inv.dtype == torch.int8
        fl = _check_int(mats.cpu().numpy(), inv, flags)
        if p == 0.0:
            assert not fl.any() and torch.equal(inv, mats)  # the identity
        if p <= 0.1:
            assert not fl.any()


@pytest.mark.parametrize("S", GF2_SIZES)
def test_sampled_invertible_gf2_triples(S):
    for p in (0.0, 0.3, 1.0):
        for B in BATCHES:
            mats = env.sample_invertible_gf2(B, S, seed=S, first=FIRST, p_nonzero=p)
            inv, flags = env.invert_bases_gf2(mats)
            want, wf = ref.inverses_gf2(mats.cpu().numpy(), S)
            assert not wf.any() and not flags.any()
            assert np.array_equal(inv.cpu().numpy(), want), (p, B)


def _edge_triples(S, seed):
    edges = ref.integer_edges(S, np.random.default_rng(seed))
    E = np.stack([m for _, m, _ in edges])
    return edges, np.stack([E, np.roll(E, 1, 0), np.roll(E, 2, 0)], 1)  # every edge at A, B and C


@pytest.mark.parametrize("S", INT_SIZES)
def test_integer_edges(S):
    edges, T = _edge_triples(S, S)
    mats = torch.from_numpy(T.astype(np.int8)).to(DEV)
    inv, flags = env.invert_bases(mats)
    _check_int(T, inv, flags)
    inv_np = inv.cpu().numpy().astype(np.int64)
    for i, (label, m, has) in enumerate(edges):
        assert bool(flags[i]) == (not (has and edges[i - 1][2] and edges[i - 2][2])), label
        assert np.array_equal(inv_np[i, 0], ref.inverse_int8(m) if has else np.zeros((S, S), np.int64)), label


@pytest.mark.parametrize("S", INT_SIZES)
def test_in_place_and_at_odd_byte_offsets(S):
    mats = env.sample_unimodular(301, S, seed=7, first=3, p_nonzero=0.3)
    _, T = _edge_triples(S, 30 + S)
    both = np.concatenate([mats.cpu().numpy().astype(np.int64), T])
    n = both.shape[0]
    for offset in (1, 3, 8):
        buf = torch.zeros(n * 3 * S * S + 16, dtype=torch.int8, device=DEV)
        m = buf[offset: offset + n * 3 * S * S].view(n, 3, S, S)
        m.copy_(torch.from_numpy(both.astype(np.int8)))
        assert m.data_ptr() % 16 == offset
        inv, flags = env.invert_bases(m)
        _check_int(both, inv, flags)
        inv2, flags2 = env.invert_bases(m, out=m)  # in place, unaligned
        assert inv2.data_ptr() == m.data_ptr() and torch.equal(inv2, inv) and torch.equal(flags2, flags)
        assert not buf[:offset].any() and not buf[offset + n * 3 * S * S:].any()
    one, fl = env.invert_bases(mats[5])  # (3, S, S) as N = 1
    assert one.shape == (1, 3, S, S) and torch.equal(one[0], env.invert_bases(mats)[0][5]) and fl.shape == (1,)


@pytest.mark.parametrize("S", GF2_SIZES)
def test_gf2_random_matrices_with_junk_bits_and_in_place(S):
    rng = np.random.default_rng(40 + S)
    for B in (1, 3, 257, 3000):
        M = rng.integers(0, 2, size=(B, 3, S, S))
        M[::2] = gf2_basis_ref.sample_invertible(5, 0, len(M[::2]), S, 0.5)  # every other triple invertible, the rest random
        bits = gf2_basis_ref.mats_to_bits(M).view(np.uint32)
        junk = bits | (rng.integers(0, 1 << 32, size=bits.shape, dtype=np.uint64).astype(np.uint32) & ~np.uint32((1 << S) - 1))
        mats = torch.from_numpy(junk.view(np.int32)).to(DEV)
        inv, flags = env.invert_bases_gf2(mats)
        want, wf = ref.inverses_gf2(bits.view(np.int32), S)
        assert np.array_equal(flags.cpu().numpy(), wf) and np.array_equal(inv.cpu().numpy(), want), B
        assert not (inv.cpu().numpy().view(np.uint32) >> S).any()
        if B > 3:
            assert 0 < int((flags != 0).sum()) < B
        inv2, flags2 = env.invert_bases_gf2(mats, out=mats)
        assert torch.equal(mats, inv) and torch.equal(flags2, flags)
    one, fl = env.invert_bases_gf2(torch.from_numpy(junk[0].view(np.int32)).to(DEV))  # (3, S) as N = 1
    assert one.shape == (1, 3, S) and np.array_equal(one[0].cpu().numpy(), want[0])


@pytest.mark.parametrize("S", INT_SIZES)
def test_integer_inverses_mod_2_are_the_gf2_inverses(S):
    mats = torch.cat([env.sample_unimodular(3000, S, seed=S, p_nonzero=0.3),
                      torch.from_numpy(_edge_triples(S, S)[1].astype(np.int8)).to(DEV)])
    inv, flags = env.invert_bases(mats)
    ok = flags == 0
    assert int(ok.sum()) > 0.9 * mats.shape[0]
    w = (mats.to(torch.int64) & 1) << torch.arange(S, device=DEV)
    inv2, fl2 = env.invert_bases_gf2(w.sum(-1).to(torch.int32))
    assert not fl2[ok].any()  # det = +-1 is odd
    wi = (inv.to(torch.int64) & 1) << torch.arange(S, device=DEV)
    assert torch.equal(wi.sum(-1).to(torch.int32)[ok], inv2[ok])


@pytest.mark.parametrize("S", GF2_SIZES)
def test_change_of_basis_mod_2_and_back(S):
    """make_synthetic_demos_gf2 with the alphabet {0, 1}: tokens are residue + shift, so the round trip is byte for byte"""
    N, R = 500, 12 if S < 25 else 20
    tape, bits, _ = env.make_synthetic_demos_gf2(N, R, S, (0, 1), (0.6, 0.4), 1, seed=S, device=DEV)
    mats = env.sample_invertible_gf2(N, S, seed=S + 1, p_nonzero=0.3)
    inv, flags = env.invert_bases_gf2(mats)
    assert not flags.any()
    b2, t2 = env.change_of_basis_gf2(bits, mats, S, tape=tape, shift=1, shift_out=1)
    assert not torch.equal(b2, bits) and not torch.equal(t2, tape)
    assert torch.equal(env.change_of_basis_factors_gf2(tape, mats, S, 1, 1), t2)
    b3, t3 = env.change_of_basis_gf2(b2, inv, S, tape=t2, shift=1, shift_out=1)
    assert torch.equal(b3, bits) and torch.equal(t3, tape)
    assert torch.equal(env.change_of_basis_factors_gf2(t2, inv, S, 1), tape)


@pytest.mark.parametrize("S", INT_SIZES)
def test_solve_in_a_changed_basis_and_verify_in_the_original(S):
    """Factors moved into a random basis (shift_out 100, room for large coefficients) sum to the transformed target; with
    the inverse triple they map back to the original tape byte for byte, which sums to the original target."""
    N, R = 2000, {4: 7, 9: 23, 16: 49}[S]
    tape, slab, dflags = env.make_synthetic_demos(N, R, S, (-1, 0, 1), (0.15, 0.7, 0.15), 1, seed=S, device=DEV)
    keep = torch.nonzero(dflags == 0).flatten()  # targets the int8 slab holds exactly
    assert keep.numel() > 0.9 * N
    tape, slab = tape[:, keep].contiguous(), slab[keep].contiguous()
    n = keep.numel()
    mats = env.sample_unimodular(n, S, seed=S + 2, first=FIRST, p_nonzero=0.3)
    T2, f2 = env.change_of_basis(slab, mats, S, out_dtype=torch.int16)
    assert not (f2 & env.FLAG_RANGE).any()
    tape2, tf = env.change_of_basis_factors(tape, mats, S, 1, 100)
    inv, sf = env.invert_bases(mats)
    back, bf = env.change_of_basis_factors(tape2, inv, S, 100, 1)
    good = (tf | sf | bf) == 0
    bad = int((~good).sum())
    assert bad <= 0.05 * n, bad  # singular triples and factors beyond +-100 are rare at p = 0.3
    acc2, af = env.accumulate_demos16(tape2, S, 100)
    assert not af[tf == 0].any() and torch.equal(acc2[tf == 0], T2[tf == 0])
    g = torch.nonzero(good).flatten()
    assert torch.equal(back[:, g], tape[:, g])
    acc, _ = env.accumulate_demos16(back[:, g].contiguous(), S, 1)
    assert np.array_equal(i16_ref.slab16_to_dense(acc.cpu().numpy(), S), slab_to_dense(slab[g].cpu().numpy(), S))


def test_factor_wrappers_are_the_c_entry_points():
    """change_of_basis_factors(_gf2) make the calls change_of_basis(_gf2) make, without the slab"""
    S, N, R = 9, 257, 5
    tape, slab, _ = env.make_synthetic_demos(N, R, S, seed=1, device=DEV)
    mats = env.sample_unimodular(N, S, seed=2, p_nonzero=0.3)
    _, t_ref, f_ref = env.change_of_basis(slab, mats, S, tape=tape, shift=1, shift_out=3)
    t, f = env.change_of_basis_factors(tape, mats, S, 1, 3)
    assert torch.equal(t, t_ref) and torch.equal(f & env.FLAG_TOKEN_RANGE, f_ref & env.FLAG_TOKEN_RANGE)
    assert not (f & ~env.FLAG_TOKEN_RANGE).any()
    t1, _ = env.change_of_basis_factors(tape, mats[0], S, 1, 3)  # one shared triple
    _, t1_ref, _ = env.change_of_basis(slab, mats[0], S, tape=tape, shift=1, shift_out=3)
    assert torch.equal(t1, t1_ref)
    m2 = env.sample_invertible_gf2(N, S, seed=2)
    _, t2_ref = env.change_of_basis_gf2(env.pack_gf2(slab, S), m2, S, tape=tape, shift=1, shift_out=2)
    assert torch.equal(env.change_of_basis_factors_gf2(tape, m2, S, 1, 2), t2_ref)
    assert _lib.FLAG_SINGULAR == env.FLAG_SINGULAR == 128
