"""The mod-2 game path on a B200: every tg_*_gf2 entry point at 4, 9, 16 and 25, bit for bit against tests/gf2_ref.py,
and its agreement with the integer game path taken mod 2 (steps, leaf expansion, keys, demo targets, known
factorizations of the matrix multiplication tensors)."""
import numpy as np
import pytest
import torch

from mat_mul_b200 import datasets, env
from oracle import tg_oracle as orc
from tests import gf2_ref as ref
from tests import i16_ref
from tests.helpers import dense_to_slab, geo

pytestmark = pytest.mark.gpu

SIZES = (4, 9, 16, 25)
BATCHES = (1, 3, 257, 3000)
DEV = "cuda"


def _bits(T):
    return torch.from_numpy(ref.dense_to_bits(T)).to(DEV)


def _dense(bits, S):
    return ref.bits_to_dense(bits.cpu().numpy(), S)


def _tape(tok):
    """(..., 3S) tokens -> uint8 (..., TP)"""
    tok = np.asarray(tok)
    tp = geo(tok.shape[-1] // 3)[2]
    out = np.zeros(tok.shape[:-1] + (tp,), dtype=np.uint8)
    out[..., : tok.shape[-1]] = tok
    return torch.from_numpy(out).to(DEV)


def _states(S, B, rng, density=0.5):
    T = (rng.random((B, S, S, S)) < density).astype(np.int64)
    T[0] = 0 if B > 2 else T[0]
    return T


def _tokens(shape, S, rng):
    """any byte is a token; a third of the records use the usual alphabet [0, 2 shift]"""
    tok = rng.integers(0, 256, size=shape + (3 * S,))
    small = rng.random(shape) < 0.3
    tok[small] = rng.integers(0, 5, size=(int(small.sum()), 3 * S))
    return tok


@pytest.mark.parametrize("S", SIZES)
def test_pack_and_unpack(S):
    rng = np.random.default_rng(S)
    for B in BATCHES:
        T = rng.integers(-128, 128, size=(B, S, S, S))
        bits = env.pack_gf2(torch.from_numpy(dense_to_slab(T)).to(DEV), S)
        assert np.array_equal(bits.cpu().numpy(), ref.dense_to_bits(T)), B
        T16 = rng.integers(-32768, 32768, size=(B, S, S, S))
        bits16 = env.pack_gf2(torch.from_numpy(i16_ref.dense_to_slab16(T16)).to(DEV), S)
        assert np.array_equal(bits16.cpu().numpy(), ref.dense_to_bits(T16)), B
        slab = env.unpack_gf2(bits, S)
        assert np.array_equal(slab.cpu().numpy(), dense_to_slab(T & 1)), B
        assert torch.equal(env.expand_states(slab, S).cpu(), torch.from_numpy((T & 1).astype(np.float32)))


@pytest.mark.parametrize("S", SIZES)
@pytest.mark.parametrize("shift", (1, 2, 3, 4))
def test_step(S, shift):
    rng = np.random.default_rng(100 * S + shift)
    for B in BATCHES:
        T = _states(S, B, rng)
        tok = _tokens((B,), S, rng)
        if B > 2:
            T[1] = ref.rank1(tok[1], shift)   # solved by the step
            tok[2, :S] = shift                # u even: null
        want, wf, wn = ref.step_ref(T, tok, shift)
        bits, tape = _bits(T), _tape(tok)
        out, fl, nz = env.step_batch(bits, tape, S, shift)
        assert np.array_equal(_dense(out, S), want) and np.array_equal(fl.cpu().numpy(), wf) and np.array_equal(nz.cpu().numpy(), wn), B
        env.step_batch(bits, tape, S, shift, out=bits)  # in place
        assert torch.equal(bits, out), B


@pytest.mark.parametrize("S", SIZES)
def test_step_matches_the_integer_step_mod_2_on_demos(S):
    N, R, shift = 200, 12, 1  # |entries| <= 12: every int8 step stays in its zone
    tape, slab, fl = env.make_synthetic_demos(N, R, S, (-1, 0, 1), (0.15, 0.7, 0.15), shift, seed=S, device=DEV)
    ok = (fl & env.FLAG_RANGE) == 0
    cur, bits = slab[ok].contiguous(), env.pack_gf2(slab, S)[ok].contiguous()
    for r in reversed(range(R)):
        rec = tape[r][ok].contiguous()
        cur, f8, _ = env.step_batch(cur, rec, S, shift)
        bits, fb, nb = env.step_batch(bits, rec, S, shift)
        assert torch.equal(env.pack_gf2(cur, S), bits), r
        assert torch.equal(nb, torch.from_numpy(np.count_nonzero(_dense(bits, S).reshape(len(nb), -1), 1).astype(np.int32)).to(DEV))
    assert not bits.any() and bool((fb & env.FLAG_TERMINAL).all())


@pytest.mark.parametrize("S", SIZES)
@pytest.mark.parametrize("k", (1, 3, 8))
def test_expand_children(S, k):
    rng = np.random.default_rng(200 * S + k)
    shift = 1 + k % 4
    for B in BATCHES[:3] + (1100,):
        T = _states(S, B, rng, 0.3)
        tok = _tokens((B, k), S, rng)
        if B > 2:
            tok[1, 0] = shift  # all coefficients zero: a null child
        bits, tape = _bits(T), _tape(tok)
        kids, kf, kn, kk = env.expand_children(bits, tape, S, shift)
        nokeys = env.expand_children(bits, tape, S, shift, with_keys=False)
        assert torch.equal(nokeys[0], kids) and nokeys[3] is None
        for c in range(k):
            want, wf, wn = ref.step_ref(T, tok[:, c], shift)
            assert np.array_equal(_dense(kids[:, c].contiguous(), S), want), (B, c)
            assert np.array_equal(kf[:, c].cpu().numpy(), wf) and np.array_equal(kn[:, c].cpu().numpy(), wn), (B, c)
            assert np.array_equal(kk[:, c].cpu().numpy().view(np.uint64), ref.state_keys(want)), (B, c)
            # every child is K1 with that child's action, and keyed as the int8 slab of its values
            one, of, on = env.step_batch(bits, tape[:, c].contiguous(), S, shift)
            assert torch.equal(one, kids[:, c]) and torch.equal(of, kf[:, c]) and torch.equal(on, kn[:, c])
            assert torch.equal(env.state_keys(env.unpack_gf2(kids[:, c].contiguous(), S), S), kk[:, c])


@pytest.mark.parametrize("S", SIZES)
def test_rollout_and_replay(S):
    rng = np.random.default_rng(300 + S)
    for B in BATCHES:
        for K in (0, 1, 2, 3, 4, 5, 8, 17):
            shift = 1 + (B + K) % 4
            tape = _tokens((B, K), S, rng)
            T = _states(S, B, rng)
            for b in range(min(B, K)):  # game b is solved at step b, then more actions follow
                T[b] = np.bitwise_xor.reduce(ref.rank1(tape[b, : b + 1], shift), axis=0)
            sm = _tape(tape.transpose(1, 0, 2)) if K else torch.zeros((0, B, geo(S)[2]), dtype=torch.uint8, device=DEV)
            bits = _bits(T)
            wo, wf, wn, ws = ref.rollout_ref(T, tape, shift)
            out, fl, nz, st = env.rollout(bits, sm, S, shift)
            assert np.array_equal(_dense(out, S), wo) and np.array_equal(st.cpu().numpy(), ws), (B, K)
            assert np.array_equal(fl.cpu().numpy(), wf) and np.array_equal(nz.cpu().numpy(), wn), (B, K)
            ro, rf, rn, _ = ref.rollout_ref(T, tape, shift, freeze=False)
            out2, fl2, nz2 = env.replay(bits, sm, S, shift)
            assert np.array_equal(_dense(out2, S), ro) and np.array_equal(fl2.cpu().numpy(), rf) and np.array_equal(nz2.cpu().numpy(), rn)
            env.rollout(bits, sm, S, shift, out=bits)  # in place
            assert torch.equal(bits, out), (B, K)


@pytest.mark.parametrize("S", SIZES)
def test_state_keys_and_slice_rank(S):
    rng = np.random.default_rng(400 + S)
    for B in BATCHES:
        T = _states(S, B, rng, density=rng.choice([0.05, 0.5]))
        if B > 4:  # slices of known rank over GF(2)
            for i in range(S):
                T[1, i] = ref.with_rank(S, i % (S + 1), rng)
                T[2, i] = ref.with_rank(S, S, rng)
        bits = _bits(T)
        keys = env.state_keys(bits, S)
        assert np.array_equal(keys.cpu().numpy().view(np.uint64), ref.state_keys(T)), B
        assert torch.equal(keys, env.state_keys(env.unpack_gf2(bits, S), S)), B
        n = min(B, 300)  # the Python reference rank is slow; the rest of a large batch checks the kernel on itself
        ranks = env.slice_rank(bits, S).cpu().numpy()
        assert np.array_equal(ranks[:n], ref.slice_ranks(T[:n])), B
        if B > 4:
            assert ranks[1] == sum(i % (S + 1) for i in range(S)) and ranks[2] == S * S
        assert np.array_equal(env.slice_rank(bits[n // 2:].contiguous(), S).cpu().numpy(), ranks[n // 2:])


@pytest.mark.parametrize("S", SIZES)
def test_demo_targets_keep_their_parity(S):
    """tg_demo_accumulate keeps the low byte, tg_demo_accumulate_i16 the int16 value and tg_demo_gen_philox the low
    byte: packed, each is the mod-2 sum of the tape's terms, RANGE-flagged targets included."""
    N, R, shift = 300, 40 if S < 25 else 60, 3
    vals, probs = (-3, -2, -1, 0, 1, 2, 3), (0.1, 0.1, 0.1, 0.4, 0.1, 0.1, 0.1)
    tape, slab, fl = env.make_synthetic_demos(N, R, S, vals, probs, shift, seed=11, device=DEV)
    tok = tape.permute(1, 0, 2).cpu().numpy()[:, :, : 3 * S]
    want = np.bitwise_xor.reduce(ref.rank1(tok, shift), axis=1)
    assert bool((fl & env.FLAG_RANGE).any())  # targets beyond the int8 zone are part of the check
    assert np.array_equal(_dense(env.pack_gf2(slab, S), S), want)
    s8, f8 = env.accumulate_demos(tape, S, shift)
    assert np.array_equal(_dense(env.pack_gf2(s8, S), S), want)
    s16, _ = env.accumulate_demos16(tape, S, shift)
    assert np.array_equal(_dense(env.pack_gf2(s16, S), S), want)
    # the mod-2 replay of the demo's actions solves the packed target
    out, flags, _, steps = env.rollout(env.pack_gf2(s16, S), tape.flip(0).contiguous(), S, shift)
    assert not out.any() and bool((flags & env.FLAG_TERMINAL).all()) and not bool((flags & env.FLAG_RANGE).any())


def test_strassen_mod_2():
    uu, vv, ww = (x.cpu().numpy().astype(np.int64) for x in datasets.get_strassen_factors("cpu"))
    shift = 1
    tok = np.concatenate([uu, vv, ww], axis=1) + shift  # (7, 12)
    T = orc.build_matmul_tensor(2)[None].astype(np.int64)
    assert np.array_equal(np.einsum("ri,rj,rk->ijk", uu, vv, ww), T[0])  # the factors' convention is the tensor's
    bits = _bits(T)
    tape = _tape(tok[:, None, :])  # (7, 1, TP)
    out, flags, nnz, steps = env.rollout(bits, tape, 4, shift)
    assert not out.any() and int(flags[0]) & env.FLAG_TERMINAL and int(steps[0]) == 7 and int(nnz[0]) == 0
    assert not env.replay(bits, tape, 4, shift)[0].any()
    # six of the seven do not reach zero
    assert env.rollout(bits, tape[:6].contiguous(), 4, shift)[0].any()


@pytest.mark.parametrize("n", (3, 4, 5))
def test_naive_factorizations_mod_2(n):
    S = n * n
    T = orc.build_matmul_tensor(n)[None].astype(np.int64)
    cells = np.argwhere(T[0])  # the n^3 unit terms e_i (x) e_j (x) e_k
    assert len(cells) == n ** 3
    shift = 4
    tok = np.full((n ** 3, 3 * S), shift)
    for r, (i, j, k) in enumerate(cells):
        tok[r, i] += 1
        tok[r, S + j] -= 1  # coefficient -1: odd
        tok[r, 2 * S + k] += 3
    bits = _bits(T)
    tape = _tape(tok[:, None, :])
    out, flags, nnz, steps = env.rollout(bits, tape, S, shift)
    assert not out.any() and int(steps[0]) == n ** 3 and int(flags[0]) & env.FLAG_TERMINAL
    ranks = env.slice_rank(bits, S).cpu().numpy()
    assert ranks[0] == ref.slice_ranks(T)[0]
