"""CPU checks of the int16 game path's references (tests/i16_ref.py).  The references are pinned against the C oracle on
int8-zone inputs, where the int8 and int16 contracts coincide (argument rules: tests/test_cabi_args.py)."""
import numpy as np
import pytest

from oracle import tg_oracle as orc
from tests import i16_ref as ref
from tests.test_edges_ref import det_int, rank_int, slice_ranks

SIZES = (4, 9, 16)  # the C oracle's rollout keeps scratch tensors of at most 16^3 entries


def small_inputs(S, B, rng, lim=20, shift=2):
    T = rng.integers(-lim, lim + 1, size=(B, S, S, S))
    tok = rng.integers(0, 2 * shift + 1, size=(B, 3 * S))
    return T, tok


@pytest.mark.parametrize("S", SIZES + (25,))
def test_step_ref_matches_oracle_in_int8_zone(S):
    rng = np.random.default_rng(S)
    T, tok = small_inputs(S, 32, rng)
    T[0] = ref.rank1(tok[0], 2)  # a step to the zero tensor
    tok[1, S:2 * S] = 2          # a null action (v = 0)
    out, flags, nnz = ref.step_ref(T, tok, 2)
    want, wflags, wnnz = orc.step_batch(T, tok, 2)
    assert np.array_equal(out, want) and np.array_equal(flags, wflags) and np.array_equal(nnz, wnnz)
    assert flags[0] & ref.FLAG_TERMINAL and flags[1] & ref.FLAG_NULL and not (flags & ref.FLAG_RANGE).any()


def test_step_ref_zone_edges():
    S, shift = 4, 1
    tok = np.full((4, 12), 2)  # u = v = w = 1 everywhere: every entry drops by one
    T = np.zeros((4, S, S, S), dtype=np.int64)
    T[0, 1, 2, 3] = -16383  # -> -16384: inside
    T[1, 1, 2, 3] = -16384  # -> -16385: outside
    T[2, 1, 2, 3] = 16384   # -> 16383: inside
    T[3, 1, 2, 3] = 16385   # -> 16384: outside
    T += 1
    T[:, 1, 2, 3] -= 1
    out, flags, _ = ref.step_ref(T, tok, shift)
    assert out[:, 1, 2, 3].tolist() == [-16384, -16385, 16383, 16384]
    assert ((flags & ref.FLAG_RANGE) != 0).tolist() == [False, True, False, True]
    tok[2, 0] = 3  # over the token bound 2 * shift
    assert ref.step_ref(T, tok, shift)[1][2] & ref.FLAG_RANGE


@pytest.mark.parametrize("S", SIZES)
def test_rollout_ref_matches_oracle_in_int8_zone(S):
    rng = np.random.default_rng(10 + S)
    B, K, shift = 24, 6, 1
    tape = rng.integers(0, 3, size=(B, K, 3 * S))
    T = rng.integers(-8, 9, size=(B, S, S, S))
    for b, t in ((0, 0), (1, 3), (2, K - 1)):  # games solved at step t, continued by more steps
        T[b] = ref.rank1(tape[b, : t + 1], shift).sum(0)
    T[3] = 0  # solved before the first step
    out, flags, nnz, steps = ref.rollout_ref(T, tape, shift)
    wo, wf, wn, ws = orc.rollout_batch(T, tape, shift)
    assert np.array_equal(out, wo) and np.array_equal(flags, wf) and np.array_equal(nnz, wn) and np.array_equal(steps, ws)
    assert steps[:4].tolist() == [1, 4, K, 0]
    ro, rf, rn, _ = ref.rollout_ref(T, tape, shift, freeze=False)
    for b in range(B):
        assert np.array_equal(ro[b], orc.take_actions(tape[b], T[b], shift))
    assert np.array_equal(rn, np.count_nonzero(ro.reshape(B, -1), axis=1))


def test_rollout_ref_flags_a_walk_that_crosses_the_zone_and_returns():
    S, shift = 4, 4
    tok_dn = np.array([8] * 4 + [8] * 4 + [8] * 4)  # u = v = w = 4: every entry drops by 64
    tok_up = np.array([0] * 4 + [8] * 4 + [8] * 4)  # u = -4: every entry rises by 64
    T = np.full((2, S, S, S), -16384 + 63)  # one step down reaches -16385
    tape = np.stack([np.stack([tok_dn, tok_up]), np.stack([tok_up, tok_dn])])
    out, flags, _, steps = ref.rollout_ref(T, tape, shift)
    assert np.array_equal(out, T) and steps.tolist() == [2, 2]
    assert ((flags & ref.FLAG_RANGE) != 0).tolist() == [True, False]


def test_state_key_ref_matches_python_integers_and_oracle():
    rng = np.random.default_rng(3)
    for S in (4, 9):
        T = rng.integers(-100, 101, size=(5, S, S, S))
        keys = ref.state_keys(T)
        assert [int(k) for k in keys] == [ref.state_key_int(t) for t in T]
        assert np.array_equal(keys, orc.state_key_batch(T))
    T = rng.integers(-32768, 32768, size=(3, 25, 25, 25))
    assert [int(k) for k in ref.state_keys(T)] == [ref.state_key_int(t) for t in T]
    # linear in T: the key of a rank-1 action is the product of its three factor sums (tg_expand_children's rule)
    tok = rng.integers(0, 9, size=(25 * 3,))
    A, Bc, Cc = ref.key_consts(25)
    f = [sum((int(t) - 4) * c for t, c in zip(tok[m * 25:(m + 1) * 25], K)) for m, K in enumerate((A, Bc, Cc))]
    assert ref.state_key_int(ref.rank1(tok, 4)) == (f[0] * f[1] * f[2]) & ref.M64


def test_companion_matrices_have_the_prime_determinants():
    for c in (1, 19, 61, 379):
        M = ref.companion_det(2**31 - c)
        assert det_int(M) == 2**31 - c and rank_int(M) == 4
    block = np.zeros((1, 8, 8, 8), dtype=np.int64)
    block[0, 0, :4, :4] = ref.companion_det(2**31 - 1)
    block[0, 0, 4:, 4:] = ref.companion_det(2**31 - 19)
    assert slice_ranks(block)[0] == 8


def test_slab16_round_trip():
    rng = np.random.default_rng(1)
    for S in (4, 9, 16, 25):
        T = rng.integers(-32768, 32768, size=(3, S, S, S))
        slab = ref.dense_to_slab16(T)
        assert slab.shape == (3, ref.geo(S)[1]) and np.array_equal(ref.slab16_to_dense(slab, S), T)
