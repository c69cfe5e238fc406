"""CPU checks of the mod-2 game path's reference (tests/gf2_ref.py), pinned against the C oracle (the integer game taken
mod 2) and against independent rank computations (argument rules: tests/test_cabi_args.py)."""
import ctypes as C
import itertools

import numpy as np
import pytest

from mat_mul_b200 import _lib
from oracle import tg_oracle as orc
from tests import gf2_ref as ref
from tests import oracle_any_s as orx

SIZES = (4, 9, 16, 25)


def test_layout_table():
    want = {4: (1, 16), 9: (3, 112), 16: (8, 512), 25: (20, 2000)}
    L = _lib.lib()
    rw, gb = C.c_int(), C.c_int()
    for S, w in want.items():
        assert ref.geo(S) == w
        assert L.tg_layout_gf2(S, C.byref(rw), C.byref(gb)) == 0 and (rw.value, gb.value) == w
    for S in (5, 7, 36):
        assert L.tg_layout_gf2(S, None, None) == -1


@pytest.mark.parametrize("S", SIZES)
def test_bits_round_trip_and_bit_order(S):
    rng = np.random.default_rng(S)
    T = rng.integers(-128, 128, size=(5, S, S, S))
    bits = ref.dense_to_bits(T)
    assert np.array_equal(ref.bits_to_dense(bits, S), T & 1)
    one = np.zeros((1, S, S, S), dtype=np.int64)
    i, j, k = S - 1, S // 2, S - 2
    one[0, i, j, k] = -1  # -1 is odd
    w = ref.dense_to_bits(one).view(np.uint32)[0]
    rw = ref.geo(S)[0]
    pos = i * rw + (j * S + k) // 32
    assert w[pos] == 1 << ((j * S + k) % 32) and np.count_nonzero(w) == 1


@pytest.mark.parametrize("S", SIZES)
def test_step_ref_is_the_integer_step_mod_2(S):
    rng = np.random.default_rng(20 + S)
    B, shift = 48, 2
    T = rng.integers(-20, 21, size=(B, S, S, S))
    tok = rng.integers(0, 2 * shift + 1, size=(B, 3 * S))
    T[0] = orx.rank1(tok[0], shift)   # a step to the zero tensor
    T[1] = orx.rank1(tok[1], shift) + 2 * T[1]  # zero mod 2 only
    tok[2, S:2 * S] = shift + 2 * rng.integers(-1, 2, size=S)  # v even, not zero: null mod 2 only
    out, flags, nnz = ref.step_ref(T, tok, shift)
    if S <= 16:
        want = orc.step_batch(T, tok, shift)[0]
    else:
        want = np.stack([T[b] - orx.rank1(tok[b], shift) for b in range(B)])
    assert np.array_equal(out, want & 1)
    assert np.array_equal(nnz, np.count_nonzero((want & 1).reshape(B, -1), axis=1))
    assert flags[0] & ref.FLAG_TERMINAL and flags[1] & ref.FLAG_TERMINAL and flags[2] & ref.FLAG_NULL
    assert np.array_equal(out[2], T[2] & 1)


def test_tokens_take_any_byte():
    S = 4
    tok = np.array([[255, 0, 3, 128] + [7] * 4 + [9] * 4])  # shift 3: coefficients 252, -3, 0, 125, 4, 6
    u, v, w = ref.factors_mod2(tok, 3)
    assert u.tolist() == [[0, 1, 0, 1]] and not v.any() and not w.any()


@pytest.mark.parametrize("S", SIZES)
def test_replay_and_rollout_ref(S):
    rng = np.random.default_rng(30 + S)
    B, K, shift = 16, 6, 1
    tape = rng.integers(0, 3, size=(B, K, 3 * S))
    T = rng.integers(-8, 9, size=(B, S, S, S))
    for b, t in ((0, 0), (1, 3), (2, K - 1)):  # solved mod 2 at step t, continued by more steps
        T[b] = ref.rank1(tape[b, : t + 1], shift).sum(0)
    T[3] = 2  # zero mod 2 before the first step
    ro, rf, rn, _ = ref.rollout_ref(T, tape, shift, freeze=False)
    for b in range(B):
        want = orc.take_actions(tape[b], T[b], shift) if S <= 16 else T[b] - sum(orx.rank1(t, shift) for t in tape[b])
        assert np.array_equal(ro[b], want & 1)
    out, flags, nnz, steps = ref.rollout_ref(T, tape, shift)
    assert steps[:4].tolist() == [1, 4, K, 0]
    assert (flags[:4] & ref.FLAG_TERMINAL).all() and not nnz[:4].any()
    for b in range(B):  # a frozen game is the replay of its first steps[b] actions
        assert np.array_equal(out[b], ref.rollout_ref(T[b:b + 1], tape[b:b + 1, : steps[b]], shift, freeze=False)[0][0])


def test_state_key_ref_is_the_int8_key_of_the_values():
    rng = np.random.default_rng(4)
    for S in (4, 9, 16):
        T = rng.integers(-3, 4, size=(6, S, S, S))
        assert np.array_equal(ref.state_keys(T), orc.state_key_batch(T & 1))
    assert ref.state_keys(np.zeros((1, 25, 25, 25)))[0] == 0


@pytest.mark.parametrize("S", SIZES)
def test_rank_gf2_on_matrices_of_known_rank(S):
    rng = np.random.default_rng(40 + S)
    for r in sorted({0, 1, 2, S // 2, S - 1, S}):
        M = ref.with_rank(S, r, rng)
        assert ref.rank_gf2(M) == r
        assert ref.rank_gf2(M + 2 * rng.integers(-3, 4, size=M.shape)) == r  # even parts do not count


@pytest.mark.parametrize("S", (4, 9))
def test_rank_gf2_by_rowspace_enumeration(S):
    rng = np.random.default_rng(50 + S)
    for _ in range(6):
        M = rng.integers(0, 2, size=(S, S)) * (rng.random((S, 1)) < 0.7)
        rows = [int("".join(map(str, r)), 2) for r in M]
        span = set()
        for sel in itertools.product((0, 1), repeat=S):
            x = 0
            for s, row in zip(sel, rows):
                if s:
                    x ^= row
            span.add(x)
        assert len(span) == 2 ** ref.rank_gf2(M)


def test_slice_ranks_of_the_matmul_tensors():
    for n in (2, 3):
        T = orc.build_matmul_tensor(n)[None]
        # slice i = (a, b) of A: the n x n^2 block pattern has rank n over any field
        assert ref.slice_ranks(T)[0] == n ** 2 * n
