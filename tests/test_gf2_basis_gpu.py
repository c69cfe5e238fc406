"""The change of basis over GF(2) on a B200: tg_change_of_basis_gf2, tg_change_of_basis_factors_gf2 and
tg_sample_invertible_gf2 at 4, 9, 16 and 25, bit for bit against tests/gf2_basis_ref.py, against the integer change of
basis and unimodular sampler taken mod 2, and end to end: transformed demos and known factorizations still solve their
transformed tensors under the mod-2 game."""
import numpy as np
import pytest
import torch

from mat_mul_b200 import _lib, datasets, env
from oracle import tg_oracle as orc
from tests import gf2_basis_ref as ref
from tests import gf2_ref
from tests.helpers import geo, tape3_to_tokens, tokens_to_tape3

pytestmark = pytest.mark.gpu

SIZES = (4, 9, 16, 25)
BATCHES = (1, 3, 257, 3000)
PROBS = (0.0, 1 / 128, 0.3, 1.0)
FIRST = (1 << 32) - 2
DEV = "cuda"


def _bits(T):
    return torch.from_numpy(gf2_ref.dense_to_bits(T)).to(DEV)


def _dense(bits, S):
    return gf2_ref.bits_to_dense(bits.cpu().numpy(), S)  # asserts zero padding bits and words


def _random_mats(n, S, rng, junk=True):
    """int32 (n, 3, S) bit matrices of random 0/1 matrices, with garbage in bits S to 31 of every row"""
    M = rng.integers(0, 2, size=(n, 3, S, S))
    bits = ref.mats_to_bits(M).view(np.uint32)
    if junk:
        bits = bits | (rng.integers(0, 1 << 32, size=bits.shape, dtype=np.uint64).astype(np.uint32) & ~np.uint32((1 << S) - 1))
    return M, bits.view(np.int32)


def _random_bits(N, S, gen):
    """N random games as a bit slab on the device (padding cleared through the 0/1 int8 slab)"""
    w = torch.randint(-(1 << 31), 1 << 31, (N, env.layout_gf2(S).game_words), generator=gen, device=DEV, dtype=torch.int64)
    return env.pack_gf2(env.unpack_gf2((w & 0xFFFFFFFF).to(torch.int32), S), S)


def _pack_residues(m8):
    """int8 (n, 3, S, S) integer matrices on the device -> int32 (n, 3, S) bit matrices of their residues"""
    S = m8.shape[-1]
    w = (m8.to(torch.int64) & 1) << torch.arange(S, device=m8.device)
    return w.sum(-1).to(torch.int32)


@pytest.mark.parametrize("S", SIZES)
def test_transform(S):
    rng = np.random.default_rng(S)
    for B in BATCHES:
        T = rng.integers(0, 2, size=(B, S, S, S))
        M, mb = _random_mats(B, S, rng)
        bits, mats = _bits(T), torch.from_numpy(mb).to(DEV)
        out = env.change_of_basis_gf2(bits, mats, S)
        assert np.array_equal(_dense(out, S), ref.transform(T, M)), B
        shared = env.change_of_basis_gf2(bits, mats[1 % B], S)  # one (3, S) triple for every game
        assert np.array_equal(_dense(shared, S), ref.transform(T, M[1 % B][None])), B
        env.change_of_basis_gf2(bits, mats, S, out=bits)  # in place
        assert torch.equal(bits, out), B


@pytest.mark.parametrize("S", SIZES)
@pytest.mark.parametrize("offset", (4, 8))
def test_transform_with_matrices_at_a_byte_offset(S, offset):
    rng = np.random.default_rng(50 + S + offset)
    B = 257
    T = rng.integers(0, 2, size=(B, S, S, S))
    M, mb = _random_mats(B, S, rng)
    buf = torch.zeros(B * 3 * S + 4, dtype=torch.int32, device=DEV)
    mats = buf[offset // 4: offset // 4 + B * 3 * S].view(B, 3, S)
    mats.copy_(torch.from_numpy(mb))
    assert mats.data_ptr() % 16 == offset % 16
    assert np.array_equal(_dense(env.change_of_basis_gf2(_bits(T), mats, S), S), ref.transform(T, M))
    shared = buf[offset // 4: offset // 4 + 3 * S].view(3, S)
    assert np.array_equal(_dense(env.change_of_basis_gf2(_bits(T), shared, S), S), ref.transform(T, M[:1]))


@pytest.mark.parametrize("S", SIZES)
def test_transform_over_more_than_one_wave_of_ctas(S):
    """More games than eight resident CTAs per SM hold: the CTAs loop over batches of games."""
    gpc = 256 // S
    N = 2 * 8 * torch.cuda.get_device_properties(0).multi_processor_count * gpc + 7
    gen = torch.Generator(device=DEV).manual_seed(S)
    bits = _random_bits(N, S, gen)
    rng = np.random.default_rng(60 + S)
    M, mb = _random_mats(N, S, rng)
    out = env.change_of_basis_gf2(bits, torch.from_numpy(mb).to(DEV), S)
    wave = N // 2
    idx = np.r_[0:40, wave - 40: wave + 40, N - 40: N]
    sel = torch.from_numpy(idx).to(DEV)
    assert np.array_equal(_dense(out[sel], S), ref.transform(_dense(bits[sel], S), M[idx]))
    env.change_of_basis_gf2(bits, torch.from_numpy(mb).to(DEV), S, out=bits)
    assert torch.equal(bits, out)


def _tape_tokens(N, R, S, rng):
    tok = rng.integers(0, 256, size=(N, R, 3 * S))
    return tok, torch.from_numpy(tokens_to_tape3(tok)).to(DEV)


@pytest.mark.parametrize("S", SIZES)
@pytest.mark.parametrize("R", (1, 23, 49))
def test_factors(S, R):
    rng = np.random.default_rng(70 + S + R)
    N = 300
    tok, tape = _tape_tokens(N, R, S, rng)
    M, mb = _random_mats(N, S, rng)
    mats = torch.from_numpy(mb).to(DEV)
    bits = _bits(rng.integers(0, 2, size=(N, S, S, S)))
    for shift_in in (1, 2, 3, 4):
        for shift_out in (1, 2, 3, 4):
            _, t2 = env.change_of_basis_gf2(bits, mats, S, tape=tape, shift=shift_in, shift_out=shift_out)
            got = tape3_to_tokens(t2.cpu().numpy(), S)  # asserts zero padding bytes
            assert np.array_equal(got, ref.factors(tok, M, shift_in, shift_out)), (shift_in, shift_out)
    _, t2 = env.change_of_basis_gf2(bits, mats[0], S, tape=tape, shift=2, shift_out=3)  # shared triple
    assert np.array_equal(tape3_to_tokens(t2.cpu().numpy(), S), ref.factors(tok, M[:1], 2, 3))


@pytest.mark.parametrize("S", SIZES)
def test_factors_with_a_shard_stride_and_in_place(S):
    """A rank's shard of a larger tape: step strides above N TP on both sides, the rows beyond the shard untouched."""
    rng = np.random.default_rng(80 + S)
    N, R, tp = 257, 23, geo(S)[2]
    tok, _ = _tape_tokens(N + 5, R, S, rng)
    big_in = torch.from_numpy(tokens_to_tape3(tok)).to(DEV)                # (R, N + 5, TP): the shard is games 0 .. N - 1
    big_out = torch.full((R, N + 9, tp), 0xAB, dtype=torch.uint8, device=DEV)
    M, mb = _random_mats(N, S, rng)
    mats = torch.from_numpy(mb).to(DEV)
    L, st = _lib.lib(), env._stream()
    _lib.check(L.tg_change_of_basis_factors_gf2(big_in.data_ptr(), (N + 5) * tp, 3, mats.data_ptr(), 1, big_out.data_ptr(),
                                                (N + 9) * tp, 1, N, R, S, st), "factors")
    want = ref.factors(tok[:N], M, 3, 1)
    assert np.array_equal(tape3_to_tokens(big_out[:, :N].cpu().numpy(), S), want)
    assert bool((big_out[:, N:] == 0xAB).all())
    _lib.check(L.tg_change_of_basis_factors_gf2(big_in.data_ptr(), (N + 5) * tp, 3, mats.data_ptr(), 1, big_in.data_ptr(),
                                                (N + 5) * tp, 1, N, R, S, st), "factors in place")
    assert np.array_equal(tape3_to_tokens(big_in[:, :N].cpu().numpy(), S), want)
    assert np.array_equal(tape3_to_tokens(big_in[:, N:].cpu().numpy(), S), tok[N:])


@pytest.mark.parametrize("S", SIZES)
def test_sampler(S):
    for p in PROBS:
        got = env.sample_invertible_gf2(300, S, seed=0xC0FFEE12345, first=FIRST, p_nonzero=p)
        want = ref.mats_to_bits(ref.sample_invertible(0xC0FFEE12345, FIRST, 300, S, p))
        assert np.array_equal(got.cpu().numpy(), want), p
        if S <= 16:  # the unimodular sampler of the same arguments, mod 2
            big = env.sample_invertible_gf2(5000, S, seed=3, first=FIRST, p_nonzero=p)
            assert torch.equal(big, _pack_residues(env.sample_unimodular(5000, S, seed=3, first=FIRST, p_nonzero=p))), p


@pytest.mark.parametrize("S", (4, 9, 16))
def test_agrees_with_the_integer_change_of_basis_mod_2(S):
    gen = torch.Generator(device=DEV).manual_seed(90 + S)
    for N in (1, 257, 3000):
        bits = _random_bits(N, S, gen)
        m8 = env.sample_unimodular(N, S, seed=S, first=11, p_nonzero=0.3)
        s8, _ = env.change_of_basis(env.unpack_gf2(bits, S), m8, S)  # int8 stores the low byte of every exact entry
        mats = env.sample_invertible_gf2(N, S, seed=S, first=11, p_nonzero=0.3)
        assert torch.equal(mats, _pack_residues(m8))
        assert torch.equal(env.pack_gf2(s8, S), env.change_of_basis_gf2(bits, mats, S)), N


@pytest.mark.parametrize("S", SIZES)
def test_transformed_demos_replay_to_zero(S):
    N, R, shift, shift_out = 500, 12 if S < 25 else 20, 1, 3
    tape, slab, _ = env.make_synthetic_demos(N, R, S, (-1, 0, 1), (0.15, 0.7, 0.15), shift, seed=S, device=DEV)
    bits = env.pack_gf2(slab, S)  # the demo targets keep their parity in the int8 slab
    mats = env.sample_invertible_gf2(N, S, seed=S + 1, p_nonzero=0.3)
    b2, t2 = env.change_of_basis_gf2(bits, mats, S, tape=tape, shift=shift, shift_out=shift_out)
    assert not torch.equal(b2, bits)
    out, flags, nnz = env.replay(b2, t2, S, shift_out)
    assert not out.any() and bool((flags & env.FLAG_TERMINAL).all()) and not nnz.any()


def _solves(T, tok, S, shift, n_terms, seed):
    """T and its n_terms factors (tokens, shift): transformed by one sampled triple, the factors still solve T' mod 2
    in exactly n_terms steps"""
    mats = env.sample_invertible_gf2(1, S, seed=seed, p_nonzero=0.5)
    bits = _bits(T[None])
    tape = torch.from_numpy(tokens_to_tape3(tok[None])).to(DEV)  # (n_terms, 1, TP)
    b2, t2 = env.change_of_basis_gf2(bits, mats, S, tape=tape, shift=shift, shift_out=2)
    assert not torch.equal(b2, bits)
    out, flags, nnz, steps = env.rollout(b2, t2, S, 2)
    assert not out.any() and int(flags[0]) & env.FLAG_TERMINAL and int(steps[0]) == n_terms


def test_strassen_still_solves_its_transformed_tensor():
    uu, vv, ww = (x.cpu().numpy().astype(np.int64) for x in datasets.get_strassen_factors("cpu"))
    tok = np.concatenate([uu, vv, ww], axis=1) + 1
    for seed in range(4):
        _solves(orc.build_matmul_tensor(2).astype(np.int64), tok, 4, 1, 7, seed)


@pytest.mark.parametrize("n", (3, 4, 5))
def test_naive_factorizations_still_solve_their_transformed_tensors(n):
    S, shift = n * n, 4
    T = orc.build_matmul_tensor(n).astype(np.int64)
    cells = np.argwhere(T)
    tok = np.full((n ** 3, 3 * S), shift)
    for r, (i, j, k) in enumerate(cells):
        tok[r, i] += 1
        tok[r, S + j] -= 1
        tok[r, 2 * S + k] += 3
    _solves(T, tok, S, shift, n ** 3, n)
