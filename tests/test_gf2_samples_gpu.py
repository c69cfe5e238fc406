"""The mod-2 training samples on a B200: tg_demo_sample_gf2 and tg_expand_f32_gf2 at 4, 9, 16 and 25, bit for bit against
tests/gf2_samples_ref.py, against the integer batcher taken mod 2, end to end from generated demos, and through env."""
import ctypes as C

import numpy as np
import pytest
import torch

from mat_mul_b200 import _lib, env
from tests import gf2_ref
from tests import gf2_samples_ref as ref
from tests.helpers import geo

pytestmark = pytest.mark.gpu

SIZES = (4, 9, 16, 25)
SHIFTS = (0, 1, 2, 8)
DEV = "cuda"
V5, P5 = (-2, -1, 0, 1, 2), (0.05, 0.10, 0.70, 0.10, 0.05)
SENTINEL = -7.0


def _records(tok):
    """tokens (N, R, 3S) -> demo-major records uint8 (N, R, TP) on the device"""
    N, R, S3 = tok.shape
    rec = np.zeros((N, R, geo(S3 // 3)[2]), dtype=np.uint8)
    rec[..., :S3] = tok
    return torch.from_numpy(rec).to(DEV)


def _indices(N, R, nb, rng):
    """nb indices: a = 0, a = R - 1 and out-of-range ones among random in-range ones"""
    idx = rng.integers(0, N * R, size=nb)
    special = [0, R - 1, N * R - 1, (N - 1) * R, -1, N * R, 1 << 40, -(1 << 40)]
    pos = rng.permutation(nb)[: min(nb, len(special))]
    idx[pos] = special[: len(pos)]
    return torch.from_numpy(idx.astype(np.int64)).to(DEV)


def _sample(records, bits, S, dim_t, replay_shift, idx, offset=0):
    """tg_demo_sample_gf2 into states that start `offset` floats into a buffer of sentinels; scalars, actions and rewards
    are prefilled with sentinels too.  Returns (states, scalars, actions, rewards, buffer)."""
    N, R = records.shape[:2]
    nb = idx.numel()
    n = nb * dim_t * S ** 3
    buf = torch.full((n + offset + 5,), SENTINEL, dtype=torch.float32, device=DEV)
    states = buf[offset:offset + n].view(nb, dim_t, S, S, S)
    scalars = torch.full((nb, 1), SENTINEL, dtype=torch.float32, device=DEV)
    actions = torch.full((nb, 3 * S), -7, dtype=torch.int64, device=DEV)
    rewards = torch.full((nb, 1), SENTINEL, dtype=torch.float32, device=DEV)
    p = lambda t: C.c_void_p(t.data_ptr())
    rc = _lib.lib().tg_demo_sample_gf2(p(records), p(bits), N, R, S, dim_t, replay_shift, p(idx), nb, p(states), p(scalars),
                                       p(actions), p(rewards), env._stream())
    assert rc == 0, rc
    return states, scalars, actions, rewards, buf


def _check(tok, targets, records, bits, S, dim_t, replay_shift, idx, offset=0):
    states, scalars, actions, rewards, buf = _sample(records, bits, S, dim_t, replay_shift, idx, offset)
    want, wsc, wac, wrw, valid = ref.samples(tok, targets, idx.cpu().numpy(), dim_t, replay_shift)
    assert bool(((states == 0) | (states == 1)).all())
    got = states.to(torch.uint8).cpu().numpy()
    bad = np.flatnonzero((got != want).reshape(len(want), -1).any(1))
    assert not len(bad), f"{len(bad)} samples differ, first {bad[:5]}"
    n = states.numel()
    assert bool((buf[:offset] == SENTINEL).all()) and bool((buf[offset + n:] == SENTINEL).all())
    v = torch.from_numpy(valid).to(DEV)
    assert np.array_equal(scalars.cpu().numpy()[valid], wsc[valid]) and np.array_equal(rewards.cpu().numpy()[valid], wrw[valid])
    assert np.array_equal(actions.cpu().numpy()[valid], wac[valid])
    assert bool((scalars[~v] == SENTINEL).all()) and bool((rewards[~v] == SENTINEL).all()) and bool((actions[~v] == -7).all())


def _store(S, N, R, rng, tokmax=256):
    tok = rng.integers(0, tokmax, size=(N, R, 3 * S))
    targets = rng.integers(0, 2, size=(N, S, S, S))
    return tok, targets, _records(tok), torch.from_numpy(gf2_ref.dense_to_bits(targets)).to(DEV)


@pytest.mark.parametrize("S", SIZES)
def test_samples_bit_for_bit(S):
    rng = np.random.default_rng(S)
    for R in (1, 7, 23) + ((100,) if S == 25 else ()):
        N = 11
        tok, targets, records, bits = _store(S, N, R, rng)
        for dim_t in (1, 2, 4, R + 2):
            for replay_shift in SHIFTS:
                nb = 257 if 257 * dim_t * S ** 3 <= 1 << 26 else max(3, (1 << 26) // (dim_t * S ** 3))
                _check(tok, targets, records, bits, S, dim_t, replay_shift, _indices(N, R, nb, rng), offset=replay_shift % 2)


@pytest.mark.parametrize("S", SIZES)
def test_batch_sizes_and_odd_offsets(S):
    rng = np.random.default_rng(100 + S)
    N, R = 40, 7
    tok, targets, records, bits = _store(S, N, R, rng)
    for nb in (1, 3, 257, 5000):
        for offset in (0, 1, 3):
            _check(tok, targets, records, bits, S, 2, 1, _indices(N, R, nb, rng), offset)


@pytest.mark.parametrize("S", SIZES)
def test_more_than_one_wave(S):
    """more state slots than the persistent grid's warps hold at once (8 CTAs of 8 warps per SM), so warps loop"""
    rng = np.random.default_rng(200 + S)
    N, R, dim_t = 64, 5, 2
    tok, targets, records, bits = _store(S, N, R, rng)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    upw = {4: 32, 9: 3, 16: 2, 25: 1}[S]
    nb = (8 * 8 * sms * upw) // dim_t + 1001
    _check(tok, targets, records, bits, S, dim_t, 2, _indices(N, R, nb, rng), offset=1)


@pytest.mark.parametrize("S", SIZES)
def test_against_the_integer_batcher(S):
    """dim_t > R on short demos: the integer batcher stages dim_t slots per sample in shared memory and refuses long ones"""
    rng = np.random.default_rng(300 + S)
    N, shift = 24, 2
    for R, dims in ((23, (1, 2, 4)), (3, (5,))):
        tape, _, _ = env.make_synthetic_demos(N, R, S, V5, P5, shift, seed=S, device=DEV)
        slab16, _ = env.accumulate_demos16(tape, S, shift)
        integer = env.DemoStore.from_tape(tape, slab16, S, shift)
        mod2 = env.DemoStore(integer.records, env.pack_gf2(slab16, S), S, shift)
        for dim_t, replay_shift in ((d, r) for d in dims for r in SHIFTS):
            idx = _indices(N, R, 300, rng)
            idx = idx[(idx >= 0) & (idx < N * R)]  # out-of-range samples leave their outputs unwritten in both
            st, sc, ac, rw = integer.samples(idx, dim_t, replay_shift)
            st2, sc2, ac2, rw2 = mod2.samples(idx, dim_t, replay_shift)
            assert torch.equal(st2, (st.to(torch.int64) & 1).to(torch.float32)), (R, dim_t, replay_shift)
            for x, y in ((sc, sc2), (ac, ac2), (rw, rw2)):
                assert torch.equal(x.view(torch.uint8), y.view(torch.uint8))


@pytest.mark.parametrize("S", SIZES)
def test_end_to_end_from_generated_demos(S):
    rng = np.random.default_rng(400 + S)
    N, R, shift = 32, 9, 2
    tape, slab, _ = env.make_synthetic_demos(N, R, S, V5, P5, shift, seed=40 + S, device=DEV)
    zeros = torch.zeros((N, env.layout_gf2(S).game_words), dtype=torch.int32, device=DEV)
    by_pack = env.DemoStore.from_tape(tape, env.pack_gf2(slab, S), S, shift)
    by_replay = env.DemoStore.from_tape(tape, env.replay(zeros, tape, S, shift)[0], S, shift)
    idx = torch.from_numpy(rng.permutation(N * R)).to(DEV)
    outs = by_pack.samples(idx, 3, shift)
    for x, y in zip(outs, by_replay.samples(idx, 3, shift)):
        assert torch.equal(x, y)
    # slot 0 of sample (d, a) is the mod-2 sum of records 0 .. a of demo d
    states = outs[0][:, 0]
    inv = torch.argsort(idx)
    for a in range(R):
        prefix = env.unpack_gf2(env.replay(zeros, tape[: a + 1], S, shift)[0], S)
        want = env.expand_states(prefix, S)
        got = states[inv[torch.arange(N, device=DEV) * R + a]]
        assert torch.equal(got, want), a
    assert torch.equal(env.expand_states(env.pack_gf2(slab, S), S), env.expand_states(env.unpack_gf2(env.pack_gf2(slab, S), S), S))


@pytest.mark.parametrize("S", SIZES)
def test_expand_f32_gf2(S):
    rng = np.random.default_rng(500 + S)
    L = _lib.lib()
    S3 = S ** 3
    p = lambda t: C.c_void_p(t.data_ptr())
    for B in (1, 3, 257, 3000):
        bits = torch.from_numpy(gf2_ref.dense_to_bits(rng.integers(0, 2, size=(B, S, S, S)))).to(DEV)
        slab = env.unpack_gf2(bits, S)
        for stride, offset in ((S3, 0), (S3, 1), (S3 + 5, 3), (S3 + 8, 1)):
            n = (B - 1) * stride + S3 + offset + 7
            got = torch.full((n,), SENTINEL, dtype=torch.float32, device=DEV)
            want = got.clone()
            assert L.tg_expand_f32_gf2(p(bits), C.c_void_p(got.data_ptr() + 4 * offset), stride, B, S, env._stream()) == 0
            assert L.tg_expand_f32(p(slab), C.c_void_p(want.data_ptr() + 4 * offset), stride, B, S, env._stream()) == 0
            assert torch.equal(got, want), (B, stride, offset)  # the floats between and around the games stay sentinels
    out = env.expand_states(bits, S)
    assert torch.equal(out, env.expand_states(slab, S))


def test_demo_store_and_expand_states_take_bit_slabs():
    rng = np.random.default_rng(600)
    S, N, R = 9, 6, 5
    tok, targets, records, bits = _store(S, N, R, rng)
    store = env.DemoStore(records, bits, S, shift=1, target_bound=12345)
    assert store.target_bound == 0
    idx = torch.arange(N * R, device=DEV)
    st, sc, ac, rw = store.samples(idx, 2, replay_shift=1)
    want, wsc, wac, wrw, _ = ref.samples(tok, targets, idx.cpu().numpy(), 2, 1)
    assert np.array_equal(st.cpu().numpy(), want.astype(np.float32)) and st.shape == (N * R, 2, S, S, S)
    assert np.array_equal(sc.cpu().numpy(), wsc) and np.array_equal(ac.cpu().numpy(), wac) and np.array_equal(rw.cpu().numpy(), wrw)
    with pytest.raises(_lib.TensorGameError):
        env.DemoStore(records, bits[:, :-4].contiguous(), S, shift=1)
    with pytest.raises(_lib.TensorGameError):
        env.expand_states(bits[:, :-4].contiguous(), S)
    out = torch.full((N, S, S, S), SENTINEL, device=DEV)
    assert env.expand_states(bits, S, out=out) is out and torch.equal(out, torch.from_numpy(targets.astype(np.float32)).to(DEV))
