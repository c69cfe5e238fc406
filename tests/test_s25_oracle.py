"""The checker at 25x25x25 (5x5 matrix multiplication).  The C oracle's step, rank-1 tensor, slice rank and state key
have no size limit; its rollout, sample item and demo loops keep scratch tensors of at most 16^3 entries, so at 25 they
come from tests/oracle_any_s.py, which is pinned here to the C oracle at 4, 9 and 16 (the code the goldens pin).  At 25
both are compared with independent restatements: numpy einsum for the rank-1 tensor and the step,
numpy.linalg.matrix_rank for get_rank, and torch's own Categorical sampler for the reference's rejection loop
(utils.py:203-233).  No golden vectors of the reference exist at this size."""
import numpy as np
import torch

import pytest

from oracle import tg_oracle as orc
from tests import oracle_any_s as orx

S = 25


def rank1(tok, shift):
    u, v, w = (np.asarray(tok[m * S:(m + 1) * S], dtype=np.int64) - shift for m in range(3))
    return np.einsum("i,j,k->ijk", u, v, w)


def test_uvw_and_step_match_einsum():
    rng = np.random.default_rng(25)
    for shift in (1, 2, 4):
        B = 6
        T = rng.integers(-20, 21, size=(B, S, S, S)).astype(np.int32)
        tok = rng.integers(0, 2 * shift + 1, size=(B, 3 * S)).astype(np.int32)
        tok[0, :S] = shift  # null action: u = 0
        T[1] = rank1(tok[1], shift)  # this action solves its state
        out, flags, nnz = orc.step_batch(T, tok, shift)
        want = np.stack([T[b] - rank1(tok[b], shift) for b in range(B)])
        assert np.array_equal(out, want)
        assert np.array_equal(nnz, (want != 0).reshape(B, -1).sum(1))
        assert flags[0] & orc.FLAG_NULL and flags[1] & orc.FLAG_TERMINAL and not (flags[2:] & orc.FLAG_TERMINAL).any()
        u, v, w = (tok[2, m * S:(m + 1) * S] - shift for m in range(3))
        assert np.array_equal(orc.uvw_to_tensor(u, v, w), rank1(tok[2], shift))


def test_slice_rank_matches_numpy():
    rng = np.random.default_rng(5)
    T = np.zeros((4, S, S, S), dtype=np.int32)
    T[0] = orc.build_matmul_tensor(5)
    for r, b in ((3, 1), (11, 2)):  # sums of r random rank-1 terms: slice ranks <= r
        for _ in range(r):
            T[b] += rank1(rng.integers(0, 3, size=3 * S), 1).astype(np.int32)
    T[3] = rng.integers(-3, 4, size=(S, S, S))
    want = [sum(int(np.linalg.matrix_rank(T[b, i].astype(np.float64))) for i in range(S)) for b in range(4)]
    assert list(orc.slice_rank_batch(T)) == want
    assert want[0] == S * 5  # every slice of the 5x5 matmul tensor has rank 5
    assert int(orc.build_matmul_tensor(5).sum()) == 125


def test_rollout_is_repeated_steps():
    rng = np.random.default_rng(7)
    B, K, shift = 3, 9, 2
    tape = rng.integers(0, 2 * shift + 1, size=(B, K, 3 * S)).astype(np.int32)
    T = np.zeros((B, S, S, S), dtype=np.int32)
    for b in range(B):
        for k in range(K):
            T[b] += rank1(tape[b, k], shift).astype(np.int32)
    T[2] += 1  # never reaches zero
    out, flags, nnz, steps = orx.rollout_batch(T, tape, shift)
    assert not out[:2].any() and list(steps[:2]) == [K, K] and (flags[:2] & orc.FLAG_TERMINAL).all()
    want = T[2].astype(np.int64) - sum(rank1(tape[2, k], shift) for k in range(K))
    assert np.array_equal(out[2], want) and steps[2] == K and nnz[2] == np.count_nonzero(want)


def test_demo_getitem_restated():
    rng = np.random.default_rng(11)
    R, shift, dim_t = 6, 1, 3
    tok = rng.integers(0, 3, size=(R, 3 * S)).astype(np.int32)
    target = sum(rank1(tok[r], shift) for r in range(R)).astype(np.int32)
    for a in (0, 2, R - 1):
        state, scalar, action, reward = orx.demo_getitem(tok, target, dim_t, a, replay_shift=shift)
        head = target - sum((rank1(tok[j], shift) for j in range(a + 1, R)), np.zeros_like(target, dtype=np.int64))
        assert np.array_equal(state[0], head)
        hi = min(a + dim_t, R)
        for s in range(1, dim_t):
            j = hi - s
            assert np.array_equal(state[s], rank1(tok[j], shift)) if j >= a + 1 else not state[s].any()
        assert scalar == R - a and reward == -(a + 1) and np.array_equal(action, tok[a])


def torch_create_synthetic_demo(values, probs, n_actions, shift):
    """utils.py:203-233 restated with torch's own sampler: factors drawn u, v, w with Categorical(probs).sample([S]),
    a triple rejected iff one factor is all zero, target = sum of the accepted rank-1 tensors."""
    vals = torch.tensor(values)
    target = torch.zeros(S, S, S)
    actions = []
    for _ in range(n_actions):
        while True:
            u, v, w = (vals[torch.distributions.Categorical(torch.tensor(probs)).sample(torch.Size([S]))] for _ in range(3))
            if u.any() and v.any() and w.any():
                break
        target += torch.einsum("i,j,k->ijk", u.float(), v.float(), w.float())
        actions.append(torch.cat([u, v, w]) + shift)
    return torch.stack(actions), target


def test_demos_from_ustream_match_torch_sampler():
    values, probs, R, shift = (-1, 0, 1), (0.15, 0.7, 0.15), 4, 1
    torch.manual_seed(2025)
    want_tok, want_tgt = zip(*[torch_create_synthetic_demo(values, probs, R, shift) for _ in range(2)])
    tok, tgt, used = orx.demos_seeded(2025, values, probs, R, S, shift, 2)
    assert np.array_equal(tok, torch.stack(want_tok).numpy()) and np.array_equal(tgt, torch.stack(want_tgt).numpy().astype(np.int32))
    # the oracle's stream position is where torch's generator stands after the loop
    assert np.array_equal(orc.mt_doubles(2025, used + 1)[used], torch.rand(1, dtype=torch.float64).numpy()[0])


def test_philox_demos_keep_contract_v1():
    # the group alias tables (contract v2) hold six tilted tables; a 25-entry factor has nine groups
    assert not orc.alias_applies((-1, 0, 1), (0.15, 0.7, 0.15), S)
    assert orc.alias_applies((-1, 0, 1), (0.15, 0.7, 0.15), 16)
    tok, tgt, ex = orx.demos_philox(3, 0, 2, (-1, 0, 1), (0.15, 0.7, 0.15), 5, S, 1)
    assert ex == 0
    for n in range(2):
        assert np.array_equal(tgt[n], sum(rank1(tok[n, r], 1) for r in range(5)))
        assert all(f.any() for r in range(5) for f in (tok[n, r].reshape(3, S) - 1))


@pytest.mark.parametrize("S_", [4, 9, 16])
def test_restatement_matches_c_oracle(S_):
    """tests/oracle_any_s.py equals the golden-pinned C oracle wherever the C oracle holds the size."""
    rng = np.random.default_rng(S_)
    shift, B, K = 2, 7, 11
    tape = (rng.integers(0, 2 * shift + 1, size=(B, K, 3 * S_)) * (rng.random((B, K, 3 * S_)) < 0.4)).astype(np.int32)
    tape = tape + shift * (tape == 0)
    T = np.zeros((B, S_, S_, S_), dtype=np.int32)
    for t in range(K // 2):
        T[0] += orx.rank1(tape[0, t], shift).astype(np.int32)
    T[1:] = rng.integers(-2, 3, size=(B - 1, S_, S_, S_))
    for a, b in zip(orc.rollout_batch(T, tape, shift), orx.rollout_batch(T, tape, shift)):
        assert np.array_equal(a, b)
    assert orx.rollout_batch(T, tape, shift)[3][0] <= K // 2  # solved at the latest in the middle of its tape
    tok = tape[1]
    tgt = sum(orx.rank1(tok[r], shift) for r in range(K)).astype(np.int32)
    for dim_t, a in ((1, 0), (3, 4), (4, K - 1)):
        for x, y in zip(orc.demo_getitem(tok, tgt, dim_t, a, shift), orx.demo_getitem(tok, tgt, dim_t, a, shift)):
            assert np.array_equal(x, y)
    V6, P6 = (-3, -1, 0, 1, 2, 3), (0.1, 0.1, 0.4, 0.2, 0.1, 0.1)  # six values: contract v1 at every size
    for vals, probs, mt in ((V6, P6, 64), ((-1, 0, 1, 2, 3, 4), (0.001, 0.995, 0.001, 0.001, 0.001, 0.001), 2)):
        c = orc.demos_philox(5, 11, 6, vals, probs, 9, S_, 4, max_tries=mt)
        r = orx.demos_philox_v1(5, 11, 6, vals, probs, 9, S_, 4, max_tries=mt)
        assert np.array_equal(c[0], r[0]) and np.array_equal(c[1], r[1]) and c[2] == r[2]
    c = orc.demos_seeded(3, (-2, -1, 0, 1, 2), (0.05, 0.10, 0.70, 0.10, 0.05), 7, S_, 2, 5)
    r = orx.demos_seeded(3, (-2, -1, 0, 1, 2), (0.05, 0.10, 0.70, 0.10, 0.05), 7, S_, 2, 5)
    assert np.array_equal(c[0], r[0]) and np.array_equal(c[1], r[1]) and c[2] == r[2]


def test_philox_restatement_matches_c_block():
    rng = np.random.default_rng(0)
    ctr = rng.integers(0, 2 ** 32, size=(5, 4), dtype=np.uint64).astype(np.uint32)
    key = (0x12345678, 0x9ABCDEF0)
    got = orx.philox4x32_10(ctr[:, 0], ctr[:, 1], ctr[:, 2], ctr[:, 3], *key)
    for i in range(5):
        assert np.array_equal(np.array([g[i] for g in got], dtype=np.uint32), orc.philox4x32_10(ctr[i], np.array(key, dtype=np.uint32)))
