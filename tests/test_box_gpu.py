"""Rectangular products <n, m, p> on a B200: tg_demo_gen_box and tg_demo_gen_box_gf2 bit for bit against
tests/box_ref.py (tape, slab or bits, flags) at 4, 9, 16 and 25 for every box of a shape with n, m, p <= 5; equality with
the cubic generators at the full box where they use contract v1; and, for every shape, the embedded target solved by its
naive factorization in int8, int16 and bits, the projection, box-preserving changes of basis and the demo store."""
import numpy as np
import pytest
import torch

from mat_mul_b200 import env
from tests import box_ref
from tests.helpers import geo, slab_to_dense, tape3_to_tokens, tokens_to_tape3

pytestmark = pytest.mark.gpu

DEV = "cuda"
V3, P3 = (-1, 0, 1), (0.15, 0.7, 0.15)
V5, P5 = (-2, -1, 0, 1, 2), (0.05, 0.10, 0.70, 0.10, 0.05)
V6, P6 = (-3, -2, -1, 0, 1, 2), (0.1, 0.2, 0.15, 0.3, 0.15, 0.1)  # six values: contract v1 at every size
ALPHABETS = {"v3": (V3, P3, 1), "v5": (V5, P5, 2), "six": (V6, P6, 3)}
SHAPES = box_ref.shapes()


def boxes_of(S):
    """(1, 1, 1), the full box and every box of the table at S, in every order of (n, m, p)."""
    return sorted({(1, 1, 1), (S, S, S)} | {b for *_, S2, b in SHAPES if S2 == S})


def int8_of(t):
    return ((np.asarray(t, dtype=np.int64) + 128) % 256 - 128).astype(np.int32)


def dense_bits(bits, S):
    return slab_to_dense(env.unpack_gf2(bits, S).cpu().numpy(), S)


def check_int(S, box, values, probs, shift, N, R, seed, first, max_tries=64):
    tape, slab, fl = env.make_synthetic_demos_box(N, R, S, box, values, probs, shift, seed, first, DEV, max_tries)
    tok, tgt, ex = box_ref.demos(seed, first, N, values, probs, R, S, shift, box, max_tries)
    assert np.array_equal(tape3_to_tokens(tape.cpu().numpy(), S), tok), (S, box)
    assert np.array_equal(slab_to_dense(slab.cpu().numpy(), S), int8_of(tgt)), (S, box)
    want = np.where(ex, env.FLAG_EXHAUSTED, 0) | np.where(box_ref.range_flags(tgt), env.FLAG_RANGE, 0)
    assert np.array_equal(fl.cpu().numpy(), want.astype(np.uint8)), (S, box)
    slab2, fl2 = env.accumulate_demos(tape, S, shift)
    assert torch.equal(slab2, slab) and torch.equal(fl2 & env.FLAG_RANGE, fl & env.FLAG_RANGE)
    return tape, slab, fl, tgt


def check_gf2(S, box, values, probs, shift, N, R, seed, first, max_tries=64):
    tape, bits, fl = env.make_synthetic_demos_box_gf2(N, R, S, box, values, probs, shift, seed, first, DEV, max_tries)
    tok, tgt, ex = box_ref.demos(seed, first, N, values, probs, R, S, shift, box, max_tries, gf2=True)
    assert np.array_equal(tape3_to_tokens(tape.cpu().numpy(), S), tok), (S, box)
    assert np.array_equal(dense_bits(bits, S), tgt), (S, box)
    assert np.array_equal(fl.cpu().numpy(), np.where(ex, env.FLAG_EXHAUSTED, 0).astype(np.uint8)), (S, box)
    return tape, bits, fl


@pytest.mark.parametrize("S", box_ref.SIZES)
@pytest.mark.parametrize("name", list(ALPHABETS))
def test_every_box_bit_for_bit(S, name):
    values, probs, shift = ALPHABETS[name]
    for box in boxes_of(S):
        check_int(S, box, values, probs, shift, 37, 5, 3, 11)
        check_gf2(S, box, values, probs, shift, 37, 5, 3, 11)


@pytest.mark.parametrize("S", box_ref.SIZES)
@pytest.mark.parametrize("R", [1, 63, 64, 65, 100])
def test_term_counts_across_the_sum_paths(S, R):
    box = {4: (2, 4, 2), 9: (6, 9, 6), 16: (12, 16, 12), 25: (15, 20, 12)}[S]
    check_int(S, box, V5, P5, 2, 301, R, 7, (1 << 33) + 5)
    check_gf2(S, box, V5, P5, 2, 301, R, 7, (1 << 33) + 5)


@pytest.mark.parametrize("S", box_ref.SIZES)
def test_large_targets_resum_exactly_in_int16(S):
    tape, slab, fl, tgt = check_int(S, (S - 1, S, S - 2), (-2, -1, 1, 2), (0.25, 0.25, 0.25, 0.25), 2, 64, 70, 9, 0)
    slab16, fl16 = env.accumulate_demos16(tape, S, 2)
    rp, _, _ = geo(S)
    got = slab16.cpu().numpy()[:, : S * rp].reshape(-1, S, rp)[:, :, : S * S].reshape(-1, S, S, S)
    assert np.array_equal(got.astype(np.int64), tgt) and not fl16.any().item()
    assert (fl & env.FLAG_RANGE).any().item()


@pytest.mark.parametrize("S", box_ref.SIZES)
def test_full_box_is_the_cubic_generator_where_it_uses_v1(S):
    alphabets = [(V6, P6, 3)] + ([(V3, P3, 1), (V5, P5, 2)] if S == 25 else [])
    for values, probs, shift in alphabets:
        a = env.make_synthetic_demos_box(200, 9, S, (S, S, S), values, probs, shift, 5, 77, DEV)
        b = env.make_synthetic_demos(200, 9, S, values, probs, shift, 5, 77, DEV)
        assert all(torch.equal(x, y) for x, y in zip(a, b))
        a = env.make_synthetic_demos_box_gf2(200, 9, S, (S, S, S), values, probs, shift, 5, 77, DEV)
        b = env.make_synthetic_demos_gf2(200, 9, S, values, probs, shift, 5, 77, DEV)
        assert all(torch.equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("S", box_ref.SIZES)
def test_exhausted(S):
    rare = ((-1, 0, 1), (0.0002, 0.9996, 0.0002))
    _, _, fl, _ = check_int(S, (1, 2, 1), *rare, 1, 50, 3, 1, 0, max_tries=2)
    assert (fl & env.FLAG_EXHAUSTED).all().item()
    _, _, fl = check_gf2(S, (1, 2, 1), *rare, 1, 50, 3, 1, 0, max_tries=2)
    assert (fl & env.FLAG_EXHAUSTED).all().item()


@pytest.mark.parametrize("S", box_ref.SIZES)
def test_bits_are_the_integer_targets_mod_2(S):
    box = boxes_of(S)[len(boxes_of(S)) // 2]
    tape, slab, fl = env.make_synthetic_demos_box(500, 20, S, box, (-1, 0, 1, 3), (0.2, 0.5, 0.2, 0.1), 3, 4, 0, DEV)
    tape2, bits, fl2 = env.make_synthetic_demos_box_gf2(500, 20, S, box, (-1, 0, 1, 3), (0.2, 0.5, 0.2, 0.1), 3, 4, 0, DEV)
    assert torch.equal(tape, tape2) and torch.equal(bits, env.pack_gf2(slab, S))
    assert torch.equal(fl & env.FLAG_EXHAUSTED, fl2)


@pytest.mark.parametrize("S", box_ref.SIZES)
def test_into_a_wider_tape(S):
    box = boxes_of(S)[1]
    N, R = 40, 6
    tp, gp = geo(S)[2], geo(S)[1]
    wide = torch.zeros((R, 3 * N, tp), dtype=torch.uint8, device=DEV)
    slab = torch.zeros((3 * N, gp), dtype=torch.int8, device=DEV)
    tape, s, fl = env.make_synthetic_demos_box(N, R, S, box, V5, P5, 2, 8, 40, DEV, tape=wide[:, N: 2 * N], slab=slab[N: 2 * N])
    tok, tgt, ex = box_ref.demos(8, 40, N, V5, P5, R, S, 2, box)
    assert np.array_equal(tape3_to_tokens(wide[:, N: 2 * N].cpu().numpy(), S), tok)
    assert np.array_equal(slab_to_dense(slab[N: 2 * N].cpu().numpy(), S), int8_of(tgt))
    assert not wide[:, :N].any().item() and not wide[:, 2 * N:].any().item() and not slab[:N].any().item()


# ---------------------------------------------------------------- end to end, every shape
def naive_tape(n, m, p, S, shift, extra=False):
    F = box_ref.naive_factors(n, m, p, S)
    if extra:  # a term with entries outside the box, and its negation, played first
        t = np.zeros((3, S), dtype=np.int64)
        t[:, 0] = 1
        for f, k in enumerate((n * m, m * p, n * p)):
            if k < S:
                t[f, S - 1] = 1
        F = np.concatenate([t[None], -t[None], F])
    tok = (F.reshape(len(F), 3 * S) + shift)[None]
    return torch.from_numpy(tokens_to_tape3(tok)).to(DEV), F


@pytest.mark.parametrize("n,m,p", [s[:3] for s in SHAPES])
def test_naive_factorization_solves_the_embedded_target(n, m, p):
    S, box = env.matmul_box(n, m, p)
    T = env.matmul_tensor(n, m, p).to(DEV)
    heads = T.float()[None].contiguous()
    slabs = {"int8": env.pack_states(heads, S), "int16": env.pack_states16(heads, S)}
    slabs["bits"] = env.pack_gf2(slabs["int8"], S)
    for extra in (False, True):
        tape, F = naive_tape(n, m, p, S, 1, extra)
        for name, slab in slabs.items():
            out, flags, nnz, steps = env.rollout(slab, tape, S, 1)
            assert int(steps[0]) == n * m * p + 2 * extra and not out.any().item(), (name, extra)
            assert int(flags[0]) & env.FLAG_TERMINAL
        if extra:
            proj = env.project_to_box(tape, S, box, 1)
            f = tape3_to_tokens(proj.cpu().numpy(), S)[0].reshape(-1, 3, S) - 1
            assert not (f * ~box_ref.inside(S, box)).any()
            s16, _ = env.accumulate_demos16(proj, S, 1)
            rp = geo(S)[0]
            got = s16.cpu().numpy()[:, : S * rp].reshape(-1, S, rp)[:, :, : S * S].reshape(S, S, S)
            assert np.array_equal(got, T.cpu().numpy())


@pytest.mark.parametrize("S", [4, 9, 16, 25])
def test_box_bases_keep_box_demos_in_the_box(S):
    N, R, shift = 96, 3, 1
    for box in sorted({b for *_, S2, b in SHAPES if S2 == S}):
        outside = np.ones((S, S, S), dtype=bool)
        outside[: box[0], : box[1], : box[2]] = False
        ins = box_ref.inside(S, box)
        if S != 25:  # the change of basis over Z stops at 16
            tape, slab, _ = env.make_synthetic_demos_box(N, R, S, box, V3, P3, shift, 2, 0, DEV)
            mats = env.box_bases(env.sample_unimodular(N, S, seed=3, p_nonzero=0.1), box)
            slab2, tape2, fl = env.change_of_basis(slab, mats, S, tape, shift, shift_out=60)
            good = (fl == 0).cpu().numpy()  # no entry left the int8 slab or the tokens of shift 60
            assert good.sum() >= 8
            d2 = slab_to_dense(slab2.cpu().numpy(), S)[good]
            assert not d2[:, outside].any()
            f2 = tape3_to_tokens(tape2.cpu().numpy(), S)[good].reshape(-1, R, 3, S).astype(np.int64) - 60
            assert not (f2 * ~ins).any()
            assert np.array_equal(np.einsum("nri,nrj,nrk->nijk", f2[:, :, 0], f2[:, :, 1], f2[:, :, 2]), d2)
            inv, sfl = env.invert_bases(mats)
            assert not sfl.any().item()
            slab3, tape3, _ = env.change_of_basis(slab2, inv, S, tape2, 60, shift_out=shift)
            g = torch.from_numpy(good).to(DEV)
            assert torch.equal(slab3[g], slab[g]) and torch.equal(tape3[:, g], tape[:, g])
        tape, bits, _ = env.make_synthetic_demos_box_gf2(N, R, S, box, V3, P3, shift, 2, 0, DEV)
        mats = env.box_bases(env.sample_invertible_gf2(N, S, seed=3), box)
        bits2, tape2 = env.change_of_basis_gf2(bits, mats, S, tape, shift)
        assert not dense_bits(bits2, S)[:, outside].any()
        f2 = tape3_to_tokens(tape2.cpu().numpy(), S).reshape(-1, R, 3, S) - shift
        assert not (f2 * ~ins).any()
        z, _, _ = env.replay(bits2, tape2, S, shift)
        assert not z.any().item()
        inv, sfl = env.invert_bases_gf2(mats)
        assert not sfl.any().item()
        bits3, tape3 = env.change_of_basis_gf2(bits2, inv, S, tape2, shift)
        assert torch.equal(bits3, bits)
        want = ((tape.int() - shift) & 1) + shift
        pad = torch.zeros_like(tape, dtype=torch.bool)
        pad[..., 3 * S:] = True
        assert torch.equal(tape3.int().masked_fill(pad, 0), want.masked_fill(pad, 0))


@pytest.mark.parametrize("S", [4, 9, 16, 25])
def test_store_of_box_demos(S):
    box = boxes_of(S)[1]
    tape, slab, _ = env.make_synthetic_demos_box(64, 8, S, box, V3, P3, 1, 6, 0, DEV)
    store = env.DemoStore.from_tape(tape, slab, S, 1)
    idx = torch.arange(64 * 8, device=DEV, dtype=torch.int64)
    states, _, actions, _ = store.samples(idx, 2)
    outside = torch.ones((S, S, S), dtype=torch.bool, device=DEV)
    outside[: box[0], : box[1], : box[2]] = False
    assert not states[:, :, outside].any().item()
    tape_b, bits, _ = env.make_synthetic_demos_box_gf2(64, 8, S, box, V3, P3, 1, 6, 0, DEV)
    states, _, _, _ = env.DemoStore.from_tape(tape_b, bits, S, 1).samples(idx, 2)
    assert not states[:, :, outside].any().item()


def test_one_store_holds_several_shapes():
    S, R = 25, 10
    shapes = [s for s in SHAPES if s[3] == S][:3]
    tp, gp = geo(S)[2], geo(S)[1]
    tape = torch.zeros((R, 30 * len(shapes), tp), dtype=torch.uint8, device=DEV)
    slab = torch.zeros((30 * len(shapes), gp), dtype=torch.int8, device=DEV)
    for i, (*_, box) in enumerate(shapes):
        env.make_synthetic_demos_box(30, R, S, box, V3, P3, 1, 1, 30 * i, DEV, tape=tape[:, 30 * i: 30 * i + 30],
                                     slab=slab[30 * i: 30 * i + 30])
    for i, (*_, box) in enumerate(shapes):
        tok, tgt, _ = box_ref.demos(1, 30 * i, 30, V3, P3, R, S, 1, box)
        assert np.array_equal(tape3_to_tokens(tape[:, 30 * i: 30 * i + 30].cpu().numpy(), S), tok)
        assert np.array_equal(slab_to_dense(slab[30 * i: 30 * i + 30].cpu().numpy(), S), int8_of(tgt))
