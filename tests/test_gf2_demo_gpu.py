"""Synthetic demonstrations modulo 2 on a B200: tg_demo_gen_gf2 at 4, 9, 16 and 25 bit for bit against
tests/gf2_demo_ref.py (tape, bits, flags), the same demos as tg_demo_gen_philox where 0 is the only even value, valid mod-2
factorizations, the distribution of the factor entries, sharding, and the Python surface."""
import ctypes as C

import numpy as np
import pytest
import torch

from mat_mul_b200 import _lib, env
from tests import gf2_demo_ref as ref
from tests import gf2_ref
from tests import gf2_samples_ref as rs
from tests.helpers import geo

pytestmark = pytest.mark.gpu

SIZES = (4, 9, 16, 25)
DEV = "cuda"
V3, P3 = (-1, 0, 1), (0.15, 0.7, 0.15)
V5, P5 = (-2, -1, 0, 1, 2), (0.05, 0.10, 0.70, 0.10, 0.05)
RARE = ((-1, 0, 1), (0.0002, 0.9996, 0.0002))  # P(even) > 0.999: contract v1, and a short max_tries forces odd triples
ALPHABETS = {
    "v3": (V3, P3),
    "v5": (V5, P5),
    "01": ((0, 1), (0.6, 0.4)),
    "no0": ((-2, -1, 1, 2), (0.3, 0.2, 0.2, 0.3)),
    "six": ((-3, -2, -1, 0, 1, 2), (0.1, 0.2, 0.15, 0.3, 0.15, 0.1)),  # six values: contract v1 at every size
    "rare": RARE,
}
FIRST = (1 << 32) - 5  # d_hi changes inside the batch


def _cases(S):
    """(N, R, shift, first_demo): batches that fill neither a warp nor a CTA, and the long action lists of 16 and 25"""
    out = [(1, 1, 1, 0), (31, 7, 2, FIRST), (33, 23, 3, 0), (1007, 7, 4, FIRST)]
    if S == 16:
        out.append((65, 49, 1, FIRST))
    if S == 25:
        out.append((40, 100, 2, FIRST))
    return out


def _tokens(tape, S):
    """step-major tape (R, N, TP) -> tokens (N, R, 3S)"""
    return tape.permute(1, 0, 2)[..., : 3 * S].cpu().numpy().astype(np.int32)


@pytest.mark.parametrize("S", SIZES)
@pytest.mark.parametrize("name", ALPHABETS)
def test_bit_for_bit_against_the_restatement(S, name):
    values, probs = ALPHABETS[name]
    max_tries = 3 if name == "rare" else 64
    ex_seen = False
    for N, R, shift, first in _cases(S):
        shift = max(shift, max(abs(v) for v in values))
        seed = 1000 * S + N + R
        tape, bits, flags = env.make_synthetic_demos_gf2(N, R, S, values, probs, shift, seed=seed, first_demo=first, device=DEV,
                                                         max_tries=max_tries)
        tok, tgt, ex = ref.demos(seed, first, N, values, probs, R, S, shift, max_tries=max_tries)
        case = (N, R, shift, first)
        assert np.array_equal(_tokens(tape, S), tok), case
        assert not tape[..., 3 * S:].any(), case
        assert np.array_equal(bits.cpu().numpy(), gf2_ref.dense_to_bits(tgt)), case
        assert np.array_equal(flags.cpu().numpy(), ex.astype(np.uint8) * _lib.FLAG_EXHAUSTED), case
        ex_seen |= bool(ex.any())
    assert ex_seen == (name == "rare")


@pytest.mark.parametrize("S", SIZES)
def test_same_demos_as_the_integer_generator_where_0_is_the_only_even_value(S):
    for (values, probs), max_tries in (((V3, P3), 64), (((-1, 0, 1), (0.1, 0.8, 0.1)), 64), (((0, 1), (0.6, 0.4)), 64),
                                       (((-3, -1, 0, 1, 3), (0.1, 0.1, 0.5, 0.2, 0.1)), 64), (RARE, 3)):
        N, R, shift = 700, 23, 3
        kw = dict(seed=77 + S, first_demo=FIRST, device=DEV, max_tries=max_tries)
        tape, slab, fl = env.make_synthetic_demos(N, R, S, values, probs, shift, **kw)
        tape2, bits, fl2 = env.make_synthetic_demos_gf2(N, R, S, values, probs, shift, **kw)
        assert torch.equal(tape, tape2), values
        assert torch.equal(bits, env.pack_gf2(slab, S)), values
        assert torch.equal(fl2, fl & _lib.FLAG_EXHAUSTED), values
        assert bool((fl2 != 0).any()) == (max_tries == 3)


@pytest.mark.parametrize("S", SIZES)
def test_every_term_is_a_move_of_the_mod_2_game(S):
    """No record is NULL under tg_step_gf2 and replaying the tape from the bit target solves every demo.  With V5 the
    integer generator's demos have terms that vanish mod 2 -- what this generator is for."""
    N, R, shift = 2000, 23 if S < 25 else 49, 2
    zeros = torch.zeros((N, env.layout_gf2(S).game_words), dtype=torch.int32, device=DEV)
    for values, probs in ((V3, P3), (V5, P5)):
        tape, bits, _ = env.make_synthetic_demos_gf2(N, R, S, values, probs, shift, seed=5 + S, device=DEV)
        for r in range(R):
            _, fl, _ = env.step_batch(zeros, tape[r], S, shift)
            assert not (fl & _lib.FLAG_NULL).any(), (values, r)
        out, fl, nnz = env.replay(bits, tape, S, shift)
        assert not out.any() and (fl & _lib.FLAG_TERMINAL).all() and not nnz.any(), values
    tape, _, _ = env.make_synthetic_demos(N, R, S, V5, P5, shift, seed=5 + S, device=DEV)
    nulls = sum(int((env.step_batch(zeros, tape[r], S, shift)[1] & _lib.FLAG_NULL).ne(0).sum()) for r in range(R))
    assert nulls > 0


def test_entry_frequencies_follow_the_mod_2_conditional_marginals():
    """4x4x4, V5, 2^20 terms: entry x of a factor conditioned on an odd entry has P(x) / (1 - pe^4) if x is odd and
    P(x) (1 - pe^3) / (1 - pe^4) if x is even, pe = P(even)."""
    S, R, shift = 4, 8, 2
    N = (1 << 20) // R
    tape, _, _ = env.make_synthetic_demos_gf2(N, R, S, V5, P5, shift, seed=2024, device=DEV)
    f = tape[..., : 3 * S].to(torch.int64).flatten() - shift
    freq = torch.bincount(f + 2, minlength=5).double().cpu().numpy() / f.numel()
    p = np.array(P5)
    pe = p[np.array(V5) % 2 == 0].sum()
    want = np.where(np.array(V5) % 2 == 1, p, p * (1 - pe ** (S - 1))) / (1 - pe ** S)
    sigma = np.sqrt(want * (1 - want) / (3 * N * R))  # entries of one factor are not independent: count factors, not entries
    assert np.all(np.abs(freq - want) < 5 * sigma + 2.0 ** -12), (freq, want)


@pytest.mark.parametrize("S", SIZES)
def test_sharded_calls_equal_one_call(S):
    N, R, shift, split, NT = 1000, 7, 1, 400, 1200
    tp, gw = geo(S)[2], env.layout_gf2(S).game_words
    tape, bits, flags = env.make_synthetic_demos_gf2(N, R, S, V5, P5, 2, seed=9, first_demo=FIRST, device=DEV)
    big = torch.full((R, NT, tp), 0xAB, dtype=torch.uint8, device=DEV)
    bslab = torch.full((NT, gw), -1, dtype=torch.int32, device=DEV)
    bfl = torch.full((NT,), 0xEE, dtype=torch.uint8, device=DEV)
    v, p = np.array(V5, dtype=np.int8), np.array(P5, dtype=np.float64)
    L = _lib.lib()
    for lo, hi in ((0, split), (split, N)):
        rc = L.tg_demo_gen_gf2(C.c_uint64(9), C.c_uint64(FIRST + lo), C.c_int64(hi - lo), R, S, 2, v.ctypes.data, p.ctypes.data,
                               len(v), 64, C.c_void_p(big[0, lo].data_ptr()), C.c_int64(NT * tp), C.c_void_p(bslab[lo].data_ptr()),
                               C.c_void_p(bfl[lo:].data_ptr()), env._stream())
        assert rc == 0, rc
    assert torch.equal(big[:, :N], tape) and (big[:, N:] == 0xAB).all()
    assert torch.equal(bslab[:N], bits) and (bslab[N:] == -1).all()
    assert torch.equal(bfl[:N], flags) and (bfl[N:] == 0xEE).all()
    b = bits.cpu().numpy()
    assert np.array_equal(gf2_ref.dense_to_bits(gf2_ref.bits_to_dense(b, S)), b)  # padding bits and words zero


@pytest.mark.parametrize("S", SIZES)
def test_python_surface_and_the_store(S):
    N, R, shift = 50, 9, 2
    lay, gw = env.layout(S), env.layout_gf2(S).game_words
    tape, bits, flags = env.make_synthetic_demos_gf2(N, R, S, V5, P5, shift, seed=S, device=DEV)
    t2 = torch.empty((R, N, lay.token_pitch), dtype=torch.uint8, device=DEV)
    b2 = torch.empty((N, gw), dtype=torch.int32, device=DEV)
    t3, b3, f3 = env.make_synthetic_demos_gf2(N, R, S, V5, P5, shift, seed=S, device=DEV, tape=t2, bits=b2)
    assert t3 is t2 and b3 is b2 and torch.equal(t2, tape) and torch.equal(b2, bits) and torch.equal(f3, flags)
    assert bits.dtype == torch.int32 and bits.shape == (N, gw) and not flags.any()
    v, p = np.array(V5, dtype=np.int8), np.array(P5, dtype=np.float64)
    t4, b4 = torch.zeros_like(t2), torch.zeros_like(b2)
    rc = _lib.lib().tg_demo_gen_gf2(C.c_uint64(S), C.c_uint64(0), C.c_int64(N), R, S, shift, v.ctypes.data, p.ctypes.data, len(v), 64,
                                    C.c_void_p(t4.data_ptr()), C.c_int64(N * lay.token_pitch), C.c_void_p(b4.data_ptr()), None,
                                    env._stream())
    assert rc == 0 and torch.equal(t4, tape) and torch.equal(b4, bits)  # flags omitted
    tok = _tokens(tape, S)
    _, tgt, _ = ref.demos(S, 0, N, V5, P5, R, S, shift)
    store = env.DemoStore.from_tape(tape, bits, S, shift)
    idx = torch.from_numpy(np.random.default_rng(S).permutation(N * R)[:200]).to(DEV)
    st, sc, ac, rw = store.samples(idx, 3, replay_shift=shift)
    want, wsc, wac, wrw, valid = rs.samples(tok, tgt, idx.cpu().numpy(), 3, shift)
    assert valid.all()
    assert np.array_equal(st.cpu().numpy(), want.astype(np.float32))
    assert np.array_equal(sc.cpu().numpy().ravel(), np.asarray(wsc, dtype=np.float32).ravel())
    assert np.array_equal(ac.cpu().numpy(), wac) and np.array_equal(rw.cpu().numpy().ravel(), np.asarray(wrw, dtype=np.float32).ravel())


@pytest.mark.parametrize("S", SIZES)
def test_into_views_of_a_larger_store(S):
    """Both mod-2 generators write a shard of demos through tape[:, a:b] / bits[a:b] views of a larger store: the same
    bytes as a call on a store of their own, and nothing outside the shard."""
    N, R, shift = 40, 6, 2
    tp, gw = env.layout(S).token_pitch, env.layout_gf2(S).game_words
    for gen, box in ((env.make_synthetic_demos_gf2, ()), (env.make_synthetic_demos_box_gf2, ((S, S - 2, 2),))):
        want = gen(N, R, S, *box, V5, P5, shift, seed=S, first_demo=N, device=DEV)
        wide = torch.zeros((R, 3 * N, tp), dtype=torch.uint8, device=DEV)
        store = torch.zeros((3 * N, gw), dtype=torch.int32, device=DEV)
        got = gen(N, R, S, *box, V5, P5, shift, seed=S, first_demo=N, device=DEV, tape=wide[:, N:2 * N], bits=store[N:2 * N])
        assert torch.equal(wide[:, N:2 * N], want[0]) and torch.equal(store[N:2 * N], want[1]) and torch.equal(got[2], want[2])
        assert not wide[:, :N].any() and not wide[:, 2 * N:].any() and not store[:N].any() and not store[2 * N:].any()
