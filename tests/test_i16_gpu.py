"""The int16 game path (tg_step_i16, tg_expand_children_i16, tg_rollout_i16, tg_replay_i16, tg_state_key_i16,
tg_slice_rank_i16) and the mirrors that fall back to it, on the GPU at every size.

- Widening identity: on int8 slabs and tapes inside the int8 zone every _i16 entry point returns the int8 result
  widened, bit for bit (slab, flags, nnz, steps, keys, ranks).
- Beyond int8: change-of-basis outputs, int16 demo targets and random int16 slabs under random legal tapes, against the
  int64 references of tests/i16_ref.py (ranks against Bareiss).
- Edges of the int16 contract: results at -16385/-16384/16383/16384, over-bound tokens, walks that cross the zone,
  slices whose determinants are 31-bit primes.
- Mirrors: get_child_states, _take_actions, tensor_factorized, get_rank and _head_key on states beyond int8 against a
  float restatement of the reference's arithmetic, and on int8-range states through the int8 kernels."""
import numpy as np
import pytest
import torch

from tests import i16_ref as ref
from tests.test_edges_ref import slice_ranks

pytestmark = pytest.mark.gpu

SIZES = [4, 9, 16, 25]
RANGE, TERMINAL, NULL = 4, 1, 2


@pytest.fixture(scope="module")
def env():
    from mat_mul_b200 import env as e

    assert torch.cuda.is_available()
    return e


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def tape_of(tok):
    """(..., 3S) tokens -> uint8 (..., TP)"""
    tok = np.asarray(tok)
    S = tok.shape[-1] // 3
    out = np.zeros(tok.shape[:-1] + (ref.geo(S)[2],), dtype=np.uint8)
    out[..., : 3 * S] = tok
    return dev(out)


def slab16(T):
    return dev(ref.dense_to_slab16(T))


def dense(slab, S):
    return ref.slab16_to_dense(slab.cpu().numpy(), S)


def u64(keys):
    return keys.cpu().numpy().view(np.uint64)


# ---------------------------------------------------------------- widening identity
@pytest.mark.parametrize("S", SIZES)
def test_widening_identity(env, S):
    rng = np.random.default_rng(100 + S)
    B, k, K, shift = 37, 5, 6, 2
    T = rng.integers(-12, 13, size=(B, S, S, S))
    tok = rng.integers(0, 2 * shift + 1, size=(B, K, 3 * S))
    T[0] = ref.rank1(tok[0, 0], shift)             # solved by the first step
    T[1] = ref.rank1(tok[1, :3], shift).sum(0)     # solved by the third step
    T[2] = 0
    tok[3, :, S:2 * S] = shift                     # null actions
    s8 = torch.from_numpy(ref.dense_to_slab16(T).astype(np.int8)).cuda()
    s16 = s8.to(torch.int16)
    rec = tape_of(tok[:, 0])
    a, b = env.step_batch(s8, rec, S, shift), env.step_batch(s16, rec, S, shift)
    assert b[0].dtype == torch.int16 and torch.equal(a[0].to(torch.int16), b[0])
    assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2]) and not bool((a[1] & RANGE).any())
    kt = tape_of(tok[:, :k])
    a, b = env.expand_children(s8, kt, S, shift), env.expand_children(s16, kt, S, shift)
    assert b[0].dtype == torch.int16 and torch.equal(a[0].to(torch.int16), b[0])
    assert all(torch.equal(x, y) for x, y in zip(a[1:], b[1:]))
    a, b = env.expand_children(s8, kt, S, shift, with_keys=False), env.expand_children(s16, kt, S, shift, with_keys=False)
    assert torch.equal(a[0].to(torch.int16), b[0]) and torch.equal(a[1], b[1]) and b[3] is None
    steps_major = tape_of(np.transpose(tok, (1, 0, 2)))
    a, b = env.rollout(s8, steps_major, S, shift), env.rollout(s16, steps_major, S, shift)
    assert torch.equal(a[0].to(torch.int16), b[0]) and all(torch.equal(x, y) for x, y in zip(a[1:], b[1:]))
    assert b[3].cpu().tolist()[:3] == [1, 3, 0]
    a, b = env.replay(s8, steps_major, S, shift), env.replay(s16, steps_major, S, shift)
    assert torch.equal(a[0].to(torch.int16), b[0]) and all(torch.equal(x, y) for x, y in zip(a[1:], b[1:]))
    assert torch.equal(env.state_keys(s8, S), env.state_keys(s16, S))
    assert torch.equal(env.slice_rank(s8, S), env.slice_rank(s16, S))
    # in place
    out = s16.clone()
    env.step_batch(out, rec, S, shift, out=out)
    assert torch.equal(out, env.step_batch(s16, rec, S, shift)[0])


# ---------------------------------------------------------------- beyond int8
def beyond_int8_states(env, S, rng):
    """int16 start states: random int16 slabs, demo targets of long tapes (accumulate_demos16) and, at 4/9/16, change
    of basis outputs (tg_change_of_basis_i16)."""
    parts = [rng.integers(-16000, 16001, size=(12, S, S, S))]
    R = 120
    dt = rng.integers(0, 9, size=(6, R, 3 * S))
    slab, fl = env.accumulate_demos16(tape_of(np.transpose(dt, (1, 0, 2))), S, 4)
    t16 = dense(slab, S)
    assert np.array_equal(t16, ref.rank1(dt, 4).sum(1)) and np.abs(t16).max() > 127
    parts.append(t16)
    if S != 25:
        T8 = rng.integers(-3, 4, size=(8, S, S, S))
        mats = env.sample_unimodular(8, S, seed=S, p_nonzero=0.3)
        o16, _ = env.change_of_basis(torch.from_numpy(ref.dense_to_slab16(T8).astype(np.int8)).cuda(), mats, S, out_dtype=torch.int16)
        parts.append(dense(o16, S))
    T = np.concatenate(parts)
    return np.clip(T, ref.ZONE_LO, ref.ZONE_HI)


@pytest.mark.parametrize("S", SIZES)
def test_beyond_int8_against_reference(env, S):
    rng = np.random.default_rng(200 + S)
    T = beyond_int8_states(env, S, rng)
    B, K, k, shift = T.shape[0], 5, 3, 4
    tok = rng.integers(0, 2 * shift + 1, size=(B, K, 3 * S))
    s = slab16(T)
    out, fl, nz = env.step_batch(s, tape_of(tok[:, 0]), S, shift)
    want, wf, wn = ref.step_ref(T, tok[:, 0], shift)
    assert np.array_equal(dense(out, S), want) and np.array_equal(fl.cpu().numpy(), wf) and np.array_equal(nz.cpu().numpy(), wn)
    kids, kf, kn, kk = env.expand_children(s, tape_of(tok[:, :k]), S, shift)
    for c in range(k):
        want, wf, wn = ref.step_ref(T, tok[:, c], shift)
        assert np.array_equal(dense(kids[:, c].contiguous(), S), want)
        assert np.array_equal(kf[:, c].cpu().numpy(), wf) and np.array_equal(kn[:, c].cpu().numpy(), wn)
        assert np.array_equal(u64(kk[:, c]), ref.state_keys(want))
    sm = tape_of(np.transpose(tok, (1, 0, 2)))
    for freeze in (True, False):
        res = (env.rollout if freeze else env.replay)(s, sm, S, shift)
        wo, wf, wn, ws = ref.rollout_ref(T, tok, shift, freeze=freeze)
        assert np.array_equal(dense(res[0], S), wo) and np.array_equal(res[1].cpu().numpy(), wf)
        assert np.array_equal(res[2].cpu().numpy(), wn)
        if freeze:
            assert np.array_equal(res[3].cpu().numpy(), ws)
    assert np.array_equal(u64(env.state_keys(s, S)), ref.state_keys(T))
    n = 3 if S == 25 else B  # Bareiss in Python integers is slow at 25x25
    assert np.array_equal(env.slice_rank(s[:n], S).cpu().numpy(), slice_ranks(T[:n]))


@pytest.mark.parametrize("S", SIZES)
def test_int16_slab_ranks_low_rank_and_full_range(env, S):
    rng = np.random.default_rng(300 + S)
    # products of narrow factors keep the rank low while entries span int16
    X = rng.integers(-120, 121, size=(4, S, S, 2))
    Y = rng.integers(-120, 121, size=(4, S, 2, S))
    T = np.concatenate([np.einsum("bijr,birk->bijk", X, Y), rng.integers(-32768, 32768, size=(2, S, S, S))])
    want = slice_ranks(T).tolist()
    assert want[4:] == [S * S] * 2 and max(want[:4]) <= 2 * S
    assert env.slice_rank(slab16(T), S).cpu().numpy().tolist() == want


# ---------------------------------------------------------------- edges
@pytest.mark.parametrize("S", SIZES)
def test_zone_edges_step_and_expand(env, S):
    shift = 1
    tok = np.full((4, 3 * S), 1)
    tok[:, 0], tok[:, S], tok[:, 2 * S + S - 1] = 2, 2, 2  # u = e_0, v = e_0, w = e_{S-1}: only (0, 0, S-1) drops by one
    T = np.zeros((4, S, S, S), dtype=np.int64)
    T[:, 0, 0, S - 1] = [-16383, -16384, 16384, 16385]
    T[:, S - 1, S - 1, 0] = 7
    out, fl, nz = env.step_batch(slab16(T), tape_of(tok), S, shift)
    assert dense(out, S)[:, 0, 0, S - 1].tolist() == [-16384, -16385, 16383, 16384]
    assert ((fl.cpu().numpy() & RANGE) != 0).tolist() == [False, True, False, True]
    kids, kf, _, _ = env.expand_children(slab16(T), tape_of(tok[:, None]), S, shift)
    assert torch.equal(kids[:, 0], out) and torch.equal(kf[:, 0], fl)


@pytest.mark.parametrize("S", SIZES)
def test_over_bound_tokens_first_and_last_byte(env, S):
    rng = np.random.default_rng(400 + S)
    B, shift = 9, 2
    T = rng.integers(-16000, 16001, size=(B, S, S, S))
    tok = rng.integers(0, 2 * shift + 1, size=(B, 3 * S))
    tok[2, 0] = 2 * shift + 1
    tok[4, 3 * S - 1] = 2 * shift + 1
    tok[6, 3 * S - 1] = 255
    out, fl, _ = env.step_batch(slab16(T), tape_of(tok), S, shift)
    f = fl.cpu().numpy()
    assert [b for b in range(B) if f[b] & RANGE] == [2, 4, 6]
    ok = [b for b in range(B) if not f[b] & RANGE]
    want, wf, _ = ref.step_ref(T[ok], tok[ok], shift)
    assert np.array_equal(dense(out, S)[ok], want) and np.array_equal(f[ok], wf)
    kf = env.expand_children(slab16(T), tape_of(tok[:, None]), S, shift)[1]
    assert torch.equal(kf[:, 0], fl)


@pytest.mark.parametrize("S", SIZES)
def test_rollout_and_replay_walks_across_the_zone(env, S):
    shift = 4
    dn = np.array([8] * S + [8] + [4] * (S - 1) + [8] + [4] * (S - 1))  # u = 4, v = w = 4 e_0: (i, 0, 0) drops by 64
    up = dn.copy()
    up[:S] = 0                                                            # u = -4: (i, 0, 0) rises by 64
    T = np.ones((5, S, S, S), dtype=np.int64)
    T[:, :, 0, 0] = -16384 + 63
    T[4, :, 0, 0] = 16383 - 63
    walks = np.stack([np.stack([dn, up, up]), np.stack([up, dn, up]), np.stack([dn, dn, up]),
                      np.stack([up, up, dn]), np.stack([up, dn, dn])])
    sm = tape_of(np.transpose(walks, (1, 0, 2)))
    for freeze in (True, False):
        res = (env.rollout if freeze else env.replay)(slab16(T), sm, S, shift)
        wo, wf, wn, ws = ref.rollout_ref(T, walks, shift, freeze=freeze)
        assert np.array_equal(dense(res[0], S)[[1, 3]], wo[[1, 3]])  # the unflagged games
        assert np.array_equal(res[1].cpu().numpy(), wf)
        assert ((wf & RANGE) != 0).tolist() == [True, False, True, False, True]
    # games solved at step t and frozen there, followed by steps that would leave the zone or break the token bound
    K = 6
    for t in range(K - 1):
        tok = np.tile(dn, (3, K, 1))
        T0 = ref.rank1(tok[:, : t + 1], shift).sum(1)
        tok[1, t + 1:, 0] = 2 * shift + 1
        tok[2, t + 1:, :S] = 0
        res = env.rollout(slab16(T0), tape_of(np.transpose(tok, (1, 0, 2))), S, shift)
        assert not res[0].any() and res[3].cpu().tolist() == [t + 1] * 3 and res[1].cpu().tolist() == [TERMINAL] * 3


@pytest.mark.parametrize("S", SIZES)
def test_slice_rank_prime_determinants(env, S):
    # block-diagonal slices of 4x4 companion matrices with determinant 2^31 - c: rank over Q is full, but every prime
    # below sees a rank-deficient block until a prime not among the blocks' determinants
    cs = [1, 19, 61, 69, 85, 99, 105, 151, 159, 171, 225, 249, 295, 325, 379]
    T = np.zeros((3, S, S, S), dtype=np.int64)
    nb = S // 4
    for g in range(3):
        for i in range(S):
            for q in range(nb):
                c = cs[(g + i + q) % len(cs)] if g < 2 else cs[q % len(cs)]
                T[g, i, 4 * q:4 * q + 4, 4 * q:4 * q + 4] = ref.companion_det(2**31 - c)
            T[g, i, 4 * nb:, 4 * nb:] = np.eye(S - 4 * nb, dtype=np.int64) * (i + 1)
    assert np.array_equal(env.slice_rank(slab16(T), S).cpu().numpy(), slice_ranks(T))


# ---------------------------------------------------------------- mirrors
def reference_rank1(action, S):
    """action_to_tensor (utils.py:69-96) restated in float32 torch: coefficient = token - 1"""
    u, v, w = (action.float() - 1).split(S, dim=-1)
    return u[:, None, None] * v[None, :, None] * w[None, None, :]


@pytest.fixture
def calls(env, monkeypatch):
    """names of the C-ABI entry points called"""
    seen = []
    real = env._call

    def spy(name, *a):
        seen.append(name)
        return real(name, *a)

    monkeypatch.setattr(env, "_call", spy)
    return seen


@pytest.mark.parametrize("S", [4, 9])
def test_mirrors_beyond_int8(env, calls, S):
    import mat_mul_b200.act as act
    import mat_mul_b200.datasets as ds
    import mat_mul_b200.utils as utils

    torch.manual_seed(S)
    k = 4
    state = torch.randint(-3, 4, (1, 2, S, S, S)).float()
    state[0, 0, 0, 0, 0] = 3000.0
    state[0, 0, 1, 1, 1] = -200.0
    actions = torch.randint(0, 3, (1, k, 3 * S))
    children = act.get_child_states(state, actions)
    for i in range(k):
        want = state[0, 0] - reference_rank1(actions[0, i], S)
        assert torch.equal(children[i][0, 0], want) and torch.equal(children[i][0, 1], state[0, 0])
    assert not children.range_flags.any() and "tg_expand_children_i16" in calls
    assert act._head_key(state) == int(ref.state_keys(state[:, 0].numpy()).view(np.int64)[0])
    want_rank = sum(int(torch.linalg.matrix_rank(state[0, 0, i].double())) for i in range(S))
    assert utils.get_rank(state) == want_rank and "tg_slice_rank_i16" in calls
    assert not bool(utils.tensor_factorized(state[:, 0]))
    assert bool(utils.tensor_factorized(torch.zeros(1, 1, S, S, S)))
    assert utils.remove_null_actions(state, [children[0], state.clone()]) == [0]
    # _take_actions: a target beyond int8, and an int8 target whose replay leaves the int8 zone (redone on int16)
    seq = [torch.zeros(3 * S, dtype=torch.int64)] + [torch.randint(0, 3, (3 * S,)) for _ in range(5)]  # first: +1 everywhere
    for tgt in (state[0, 0].clone(), torch.full((S, S, S), 63.0)):
        want = tgt.clone()
        for a in seq:
            want = want - reference_rank1(a, S)
        del calls[:]
        got = ds.SyntheticDemoDataset._take_actions(seq, tgt)
        assert got.dtype == torch.float32 and torch.equal(got, want) and "tg_replay_i16" in calls
    # a child that leaves the int8 zone from an int8 parent: the int8 expansion flags it and is redone on int16
    near = torch.full((1, 1, S, S, S), 63.0)
    del calls[:]
    kids = act.get_child_states(near, torch.full((1, 1, 3 * S), 0))  # coefficient -1 everywhere: every entry rises to 64
    assert torch.equal(kids[0][0, 0], near[0, 0] - reference_rank1(torch.zeros(3 * S, dtype=torch.int64), S))
    assert calls.count("tg_expand_children") == 1 and calls.count("tg_expand_children_i16") == 1


@pytest.mark.parametrize("S", [4, 9])
def test_mirrors_on_int8_states_take_the_int8_path(env, calls, S):
    import mat_mul_b200.act as act
    import mat_mul_b200.datasets as ds
    import mat_mul_b200.utils as utils

    torch.manual_seed(10 + S)
    state = torch.randint(-5, 6, (1, 2, S, S, S)).float()
    actions = torch.randint(0, 3, (1, 3, 3 * S))
    act.get_child_states(state, actions)
    act._head_key(state)
    utils.get_rank(state)
    utils.tensor_factorized(state[:, 0])
    ds.SyntheticDemoDataset._take_actions([torch.randint(0, 3, (3 * S,)) for _ in range(3)], state[0, 0])
    assert not [c for c in calls if c.endswith("_i16")], calls
    assert {"tg_expand_children", "tg_state_key", "tg_slice_rank", "tg_rollout", "tg_replay"} <= set(calls)


def test_mirrors_raise_beyond_int16(env):
    import mat_mul_b200.act as act
    import mat_mul_b200.utils as utils

    S = 4
    state = torch.zeros(1, 1, S, S, S)
    state[0, 0, 0, 0, 0] = 16383.0
    with pytest.raises(env.TensorGameError):  # a child at 16384 leaves the int16 zone
        act.get_child_states(state, torch.full((1, 1, 3 * S), 0))
    state[0, 0, 0, 0, 0] = 40000.0
    with pytest.raises(env.TensorGameError):
        utils.get_rank(state)
    state[0, 0, 0, 0, 0] = 0.5
    with pytest.raises(env.TensorGameError):
        utils.get_rank(state)
