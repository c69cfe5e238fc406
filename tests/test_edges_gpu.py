"""Every exactness guard at its edge: constructed inputs on both sides of each hand-derived bound, against exact int64 /
Python-integer references (tests/test_edges_ref.py).  The contract asserted throughout: no TG_FLAG_RANGE => bit-exact,
and TG_FLAG_RANGE wherever the documented zone is left."""
import numpy as np
import pytest
import torch

from tests.helpers import dense_to_slab, geo, slab_to_dense, tokens_to_tape, tokens_to_tape3
from tests.test_edges_ref import (DET_P, basis_counterexample, block_diag_det_p, change_of_basis_ref, rank1_sum,
                                  slice_ranks)

pytestmark = pytest.mark.gpu

SIZES = [4, 9, 16, 25]
RANGE, TERMINAL, PATH_EXACT = 4, 1, 64


@pytest.fixture(scope="module")
def env():
    from mat_mul_b200 import env as e

    assert torch.cuda.is_available()
    return e


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def dense16(slab16, S):
    rp, _, _ = geo(S)
    return slab16.cpu().numpy()[:, : S * rp].reshape(-1, S, rp)[:, :, : S * S].reshape(-1, S, S, S).astype(np.int64)


def decode(slab, S):
    """int8 slab (B, GP) -> ((B,S,S,S) int64, padding of each game still zero).  A flagged game's bytes are unspecified
    (a carry out of an entry that left int8 may reach the padding); unflagged games must keep it zero."""
    rp, gp, _ = geo(S)
    slab = np.asarray(slab).reshape(-1, gp)
    rows = slab[:, : S * rp].reshape(len(slab), S, rp)
    clean = ~rows[:, :, S * S:].any(axis=(1, 2)) & ~slab[:, S * rp:].any(axis=1)
    return rows[:, :, : S * S].reshape(-1, S, S, S).astype(np.int64), clean


def out_of_zone(T):
    T = np.asarray(T).reshape(len(T), -1)
    return ((T < -64) | (T > 63)).any(axis=1)


# ---------------------------------------------------------------- K1 tg_step / K8 tg_expand_children
def edge_step_batch(S, shift, rng, n=48):
    """Games whose result lands on -64 / 63 everywhere it is set, plus one entry per 'edge' game on -65, 64, -128 or
    127; inputs across the full int8 range; every coefficient +-shift (the largest |u v w| the packed update allows)."""
    coef = rng.choice([-shift, shift], size=(n, 3, S)).astype(np.int64)
    coef[:, :, rng.integers(0, S)] *= rng.integers(0, 2, size=(n, 3))  # some zero coefficients too
    P = np.einsum("ni,nj,nk->nijk", coef[:, 0], coef[:, 1], coef[:, 2])
    res = rng.choice([-64, 63, -64 + shift, 63 - shift, 0], size=P.shape).astype(np.int64)
    edge = rng.choice([-65, 64, -128, 127], size=n)
    for g in range(n):
        if g % 2:  # odd games leave the zone in exactly one entry whose input is still int8
            for _ in range(200):
                i, j, k = rng.integers(0, S, 3)
                if -128 <= edge[g] + P[g, i, j, k] <= 127:
                    res[g, i, j, k] = edge[g]
                    break
    T = res + P
    bad = (T < -128) | (T > 127)
    res[bad] = -P[bad]  # inputs must be int8: those entries land on 0
    T = res + P
    tok = (coef + shift).reshape(n, 3 * S)
    return T, tok, res


@pytest.mark.parametrize("S", SIZES)
@pytest.mark.parametrize("shift", [1, 2, 3, 4])
def test_step_range_flag_at_zone_edges(env, S, shift):
    rng = np.random.default_rng(100 * S + shift)
    T, tok, want = edge_step_batch(S, shift, rng)
    out, flags, nnz = env.step_batch(dev(dense_to_slab(T)), dev(tokens_to_tape(tok)), S, shift)
    flags = flags.cpu().numpy()
    got = slab_to_dense(out.cpu().numpy(), S)
    assert np.array_equal((flags & RANGE) != 0, out_of_zone(want))
    assert (flags[1::2] & RANGE).any() and not (flags[0::2] & RANGE).any()
    ok = (flags & RANGE) == 0
    assert np.array_equal(got[ok], want[ok])
    assert np.array_equal(nnz.cpu().numpy()[ok], np.count_nonzero(want.reshape(len(want), -1), axis=1)[ok])
    # a result of exactly -128 or 127 is still exact (the step that left the zone is exact)
    assert np.array_equal(got, want)


@pytest.mark.parametrize("S", SIZES)
@pytest.mark.parametrize("bad_tok", ["2s+1", 0x80, 0xFF])
def test_step_token_bound(env, S, bad_tok):
    shift = 2
    rng = np.random.default_rng(S)
    n = 3 * 4 + 2
    T = rng.integers(-20, 21, size=(n, S, S, S))
    tok = rng.integers(0, 2 * shift + 1, size=(n, 3 * S))
    value = 2 * shift + 1 if bad_tok == "2s+1" else bad_tok
    positions = [0, S - 1, S, 2 * S - 1, 2 * S, 3 * S - 1]  # first and last byte of u, v and w
    bad_games = list(range(0, 2 * len(positions), 2))
    for g, p in zip(bad_games, positions):
        tok[g, p] = value
    tok[1, 3 * S - 1] = 2 * shift  # the largest legal token in the last byte: not flagged
    want = T - rank1_sum(tok[:, None], shift)
    out, flags, _ = env.step_batch(dev(dense_to_slab(T)), dev(tokens_to_tape(tok)), S, shift)
    flags = flags.cpu().numpy()
    got, clean = decode(out.cpu().numpy(), S)
    assert clean[flags & RANGE == 0].all()
    for g in range(n):
        if g in bad_games:
            assert flags[g] & RANGE, (g, positions[bad_games.index(g)])
        else:
            assert not flags[g] & RANGE and np.array_equal(got[g], want[g]), g  # the siblings stay exact


@pytest.mark.parametrize("S", SIZES)
@pytest.mark.parametrize("shift", [1, 4])
def test_expand_children_range_and_token_edges(env, S, shift):
    rng = np.random.default_rng(7 * S + shift)
    B, k = 6, 8
    T, tok, _ = edge_step_batch(S, shift, rng, n=B * k)
    parents = T[::k].copy()  # children of a parent share it: their results differ only by their actions
    tok = tok.reshape(B, k, 3 * S).copy()
    tok[:, 5, 3 * S - 1] = 2 * shift + 1  # child 5: a token over the bound in the last byte of w
    tok[:, 6, S - 1] = 0xFF               # child 6: in the last byte of u
    want = parents[:, None] - rank1_sum(tok.reshape(B * k, 1, 3 * S), shift).reshape(B, k, S, S, S)
    _, _, tp = geo(S)
    tape = np.zeros((B, k, tp), dtype=np.uint8)
    tape[:, :, :3 * S] = tok
    ch, flags, nnz, _ = env.expand_children(dev(dense_to_slab(parents)), dev(tape), S, shift)
    flags = flags.cpu().numpy()
    got, clean = decode(ch.cpu().numpy(), S)
    got, clean = got.reshape(B, k, S, S, S), clean.reshape(B, k)
    assert clean[flags & RANGE == 0].all()
    assert (flags[:, 5] & RANGE).all() and (flags[:, 6] & RANGE).all()
    legal = np.ones(k, dtype=bool)
    legal[[5, 6]] = False
    w = want[:, legal]
    assert np.array_equal((flags[:, legal] & RANGE) != 0, out_of_zone(w.reshape(-1, S, S, S)).reshape(B, -1))
    ok = (flags[:, legal] & RANGE) == 0
    assert np.array_equal(got[:, legal][ok], w[ok])


# ---------------------------------------------------------------- K2 tg_rollout / tg_replay
@pytest.mark.parametrize("S", SIZES)
@pytest.mark.parametrize("junk", ["over-bound", "legal"])
def test_rollout_solved_then_junk(env, S, junk):
    """A game solved at step t and followed by tokens that would leave the zone -- over-bound tokens (0xFF: the token
    check) or legal ones that walk entry (0,0,0) below -64 (the lazy range check): zero result, steps = t + 1, TERMINAL,
    no RANGE -- for t = 0 .. 7 (every position in a segment of 8 and in the ring of 4); tg_replay on the same tape flags
    RANGE."""
    shift, K = 1, (12 if junk == "over-bound" else 80)
    ts = np.arange(8)
    N = len(ts)
    if junk == "over-bound":
        tok = np.full((N, K, 3 * S), 0xFF, dtype=np.int64)
    else:  # u_0 = v_0 = w_0 = 1 (token 2 shift): every step subtracts 1 from entry (0,0,0); 70+ steps reach -70
        tok = np.full((N, K, 3 * S), shift, dtype=np.int64)
        tok[:, :, [0, S, 2 * S]] = 2 * shift
    T = np.zeros((N, S, S, S), dtype=np.int64)
    for g, t in enumerate(ts):
        tok[g, :t + 1] = shift
        for r in range(t + 1):  # e_q (x) e_q (x) e_q, q = r mod S: the residual stays non-negative and small, zero only at the end
            tok[g, r, [r % S, S + r % S, 2 * S + r % S]] = shift + 1
        T[g] = rank1_sum(tok[g:g + 1, :t + 1], shift)[0]
    tape = dev(tokens_to_tape3(tok))
    out, flags, nnz, steps = env.rollout(dev(dense_to_slab(T)), tape, S, shift)
    flags = flags.cpu().numpy()
    assert not slab_to_dense(out.cpu().numpy(), S).any()
    assert np.array_equal(steps.cpu().numpy(), ts + 1)
    assert (flags & TERMINAL).all() and not (flags & RANGE).any(), flags
    assert not nnz.cpu().numpy().any()
    _, rflags, _ = env.replay(dev(dense_to_slab(T)), tape, S, shift)
    assert (rflags.cpu().numpy() & RANGE).all()


@pytest.mark.parametrize("S", SIZES)
@pytest.mark.parametrize("shift", [1, 2, 4])
def test_rollout_walk_to_int8_edge_and_back(env, S, shift):
    """One entry walks from -64 to -128 (or 63 to 127) and back, starting at every offset in the lazy check window
    (every chk = 64 / shift^3 steps).  The excursion stays outside [-64, 63] for 2 * (64 // shift^3) - 1 >= chk
    consecutive states, so a check always falls inside it: every game is flagged, and its final state (back in the
    zone) is still the int64 rollout."""
    c3 = shift ** 3
    n_out = 64 // c3
    offsets = list(range(max(1, 64 // c3) + 1))
    games, tapes = [], []
    for start, sgn in ((-64, 1), (63, -1)):
        for off in offsets:
            K = off + 2 * n_out
            T = np.zeros((S, S, S), dtype=np.int64)
            T[0, 0, 0], T[S - 1, S - 1, S - 1] = start, 5
            tok = np.full((K, 3 * S), shift, dtype=np.int64)
            for r in range(off, K):  # out: subtract sgn * c3 (away from 0), back: add it
                away = r < off + n_out
                tok[r, 0], tok[r, S], tok[r, 2 * S] = shift + (sgn if away else -sgn) * shift, 2 * shift, 2 * shift
            games.append(T)
            tapes.append(tok)
    Kmax = max(len(t) for t in tapes)
    tok = np.stack([np.vstack([t, np.full((Kmax - len(t), 3 * S), shift)]) for t in tapes])
    T = np.stack(games)
    want = T - rank1_sum(tok, shift)
    out, flags, _, steps = env.rollout(dev(dense_to_slab(T)), dev(tokens_to_tape3(tok)), S, shift)
    flags = flags.cpu().numpy()
    assert (flags & RANGE).all(), flags
    assert not out_of_zone(want).any()
    assert (steps.cpu().numpy() == Kmax).all()


@pytest.mark.parametrize("S", SIZES)
def test_rollout_start_outside_zone_is_flagged(env, S):
    shift, K = 2, 3
    T = np.zeros((4, S, S, S), dtype=np.int64)
    T[0, 0, 0, 0], T[1, S - 1, S - 1, S - 1], T[2, 1, 0, 0], T[3, 0, 0, 0] = 64, -65, 63, -64
    tok = np.full((4, K, 3 * S), shift, dtype=np.int64)  # null actions
    out, flags, _, steps = env.rollout(dev(dense_to_slab(T)), dev(tokens_to_tape3(tok)), S, shift)
    flags = flags.cpu().numpy()
    assert list((flags & RANGE) != 0) == [True, True, False, False]
    assert np.array_equal(slab_to_dense(out.cpu().numpy(), S)[2:], T[2:])


# ---------------------------------------------------------------- K3 tg_demo_accumulate (int8)
def product_terms(t, shift):
    """(a, b, c) coefficient triples, |a|, |b|, |c| <= shift, whose products sum to t (largest products first)."""
    prods = sorted({(a * b * c, (a, b, c)) for a in range(1, shift + 1) for b in range(1, shift + 1)
                    for c in range(1, shift + 1)}, reverse=True)
    sgn, left, out = (1 if t >= 0 else -1), abs(t), []
    while left:
        p, (a, b, c) = next(x for x in prods if x[0] <= left)
        out.append((sgn * a, b, c))
        left -= p
    return out


def demo_tape(entries, R, S, shift):
    """One demo per list of ((i, j, k), value) that fits R records: records e_i (x) e_j (x) e_k scaled to sum to each
    value, the rest null records.  Returns tokens (N, R, 3S) of the demos that fit."""
    recs = [[((i, j, k), t) for (i, j, k), v in ents for t in product_terms(v, shift)] for ents in entries]
    recs = [r for r in recs if len(r) <= R]
    tok = np.full((len(recs), R, 3 * S), shift, dtype=np.int64)
    for n, rr in enumerate(recs):
        for r, ((i, j, k), (a, b, c)) in enumerate(rr):
            tok[n, r, [i, S + j, 2 * S + k]] = (shift + a, shift + b, shift + c)
    return tok


K3_CASES = [(1, 191), (1, 192), (2, 23), (2, 24), (4, 2), (4, 3)]  # R shift^3 = 191 / 192 / 184 / 192 / 128 / 192


@pytest.mark.parametrize("S", SIZES)
@pytest.mark.parametrize("shift,R", K3_CASES + [(2, 40), (4, 64), (4, 65)])
def test_accumulate_int8_final_entries_at_the_alias_edges(env, S, shift, R):
    """Final entries of +-63/64/65, +-191, 192 .. 255 and 256 + k (k in [-64, 63]: bytes that would decode back inside
    the zone), alone and next to neighbours of +-1 in the same packed word, as far as R records reach them: at R shift^3
    on both sides of 191 (where the 4x4x4 thread kernel hands over and the per-thread guard starts), at 320, and, at
    16x16x16, on both sides of the tensor-core path's R <= 64.  Two demos put one thread far above the per-thread bound
    with entries that cancel.  RANGE <=> a final entry outside [-64, 63]; unflagged demos are exact; where documented (16x16x16 with
    R <= 64, and 25x25x25) the stored byte is the exact value mod 256 even when flagged."""
    values = [0, 63, -64, 64, -65, 127, -128, 191, -191, 192, 200, 255, -192, -255, 256 - 64, 256 - 1, 256, 256 + 63,
              -256 + 63, -256 - 64, 4095, -4096]
    entries = [[((0, 0, 1), v), ((0, 0, 0), 1), ((0, 0, 2), -1)] for v in values] + [[((0, 0, 1), v)] for v in values]
    # one thread (column j = 0) far above the per-thread bound whose entries cancel, next to packed neighbours
    half = max(1, (R - 3) // 2)
    entries.append([((1, 0, 0), half * shift ** 3), ((1, 0, 0), -half * shift ** 3), ((2, 1, 1), 1), ((S - 1, S - 1, S - 1), -1)])
    entries.append([((1, 0, 0), (R // 2) * shift ** 3), ((1, 0, 0), -(R // 2) * shift ** 3)])
    tok = demo_tape(entries, R, S, shift)
    assert len(tok) >= 5
    want = rank1_sum(tok, shift)
    slab, flags = env.accumulate_demos(dev(tokens_to_tape3(tok)), S, shift)
    flags = flags.cpu().numpy()
    got, clean = decode(slab.cpu().numpy(), S)
    assert np.array_equal((flags & RANGE) != 0, out_of_zone(want)), (flags, values)
    ok = (flags & RANGE) == 0
    assert clean[ok].all() and np.array_equal(got[ok], want[ok])
    if S == 25 or (S == 16 and R <= 64):
        assert np.array_equal(got & 0xFF, want & 0xFF)


@pytest.mark.parametrize("S", SIZES)
@pytest.mark.parametrize("shift,R", K3_CASES)
def test_synthetic_demos_two_value_alphabet(env, S, shift, R):
    """make_synthetic_demos with the alphabet (-s, s) (every coefficient at its bound) against the oracle's Philox
    contract: tokens bit for bit; targets exact where unflagged and RANGE exactly where a target leaves the zone."""
    from tests import oracle_any_s as orx

    N = 16 if S == 25 else 64
    values, probs = (-shift, shift), (0.5, 0.5)
    tape, slab, flags = env.make_synthetic_demos(N, R, S, values, probs, shift, seed=11)
    if S == 25:
        tok, tgt, _ = orx.demos_philox(11, 0, N, values, probs, R, S, shift)
    else:
        from oracle import tg_oracle as orc

        tok, tgt, _ = orc.demos_philox(11, 0, N, values, probs, R, S, shift)
    assert np.array_equal(tape.cpu().numpy()[:, :, :3 * S].transpose(1, 0, 2), tok)
    want = rank1_sum(tok, shift)
    assert np.array_equal(want, np.asarray(tgt, dtype=np.int64))
    flags = flags.cpu().numpy()
    assert np.array_equal((flags & RANGE) != 0, out_of_zone(want))
    got, clean = decode(slab.cpu().numpy(), S)
    ok = (flags & RANGE) == 0
    assert clean[ok].all() and np.array_equal(got[ok], want[ok])


# ---------------------------------------------------------------- K4 tg_demo_sample / tg_demo_sample_dm
def sample_reference(tok, tgt, S, dim_t, idx, replay_shift):
    from tests import oracle_any_s as orx

    R = tok.shape[1]
    if S == 25:
        return np.stack([orx.demo_getitem(tok[i // R], tgt[i // R], dim_t, i % R, replay_shift)[0] for i in idx])
    from oracle import tg_oracle as orc

    return np.stack([orc.demo_getitem(tok[i // R], tgt[i // R], dim_t, i % R, replay_shift)[0] for i in idx])


@pytest.mark.parametrize("S", [4, 9, 16])
@pytest.mark.parametrize("R", [95, 96])
def test_demo_sample_pack16_threshold(env, S, R):
    """tg_demo_sample at 127 + R cmax^3 = 32712 (R = 95, packed 16-bit lanes) and 32839 (R = 96, int32): replay_shift 1
    turns tokens 8 into coefficient 7, so replaying every action of a demo moves an entry by R * 343 from a target of
    +-127; tokens 0 (coefficient -1) in some records give lanes of opposite sign in the same word."""
    N, dim_t = 3, 2
    rng = np.random.default_rng(R + S)
    tok = np.where(rng.random((N, R, 3 * S)) < 0.9, 8, 0).astype(np.int64)
    tok[0] = 8  # all coefficients 7: entries reach 127 - R * 343 < -32500
    tgt = rng.choice([-127, 127], size=(N, S, S, S)).astype(np.int64)
    tgt[0] = 127 if R % 2 else -128
    idx = np.concatenate([np.arange(0, N * R, R), rng.integers(0, N * R, 13)])
    want = sample_reference(tok, tgt, S, dim_t, idx, 1)
    assert np.abs(want).max() > 32000
    st, _, _, _ = env.demo_samples(dev(tokens_to_tape3(tok)), dev(dense_to_slab(tgt)), dev(idx), S, dim_t, replay_shift=1)
    assert np.array_equal(st.cpu().numpy(), want.astype(np.float32))


@pytest.mark.parametrize("S", SIZES)
@pytest.mark.parametrize("replay_shift", [0, 8])
@pytest.mark.parametrize("over", [0, 1])
def test_demo_sample_dm_int16_targets_at_the_bound(env, S, replay_shift, over):
    """tg_demo_sample_dm from int16 targets at +-target_bound with target_bound = 32767 - R cmax^3 (packed 16-bit lanes)
    and that value + 1 (int32): opposite signs in the two lanes of each pair, so a borrow between lanes would show; the
    tapes replay every coefficient at cmax = 8 (replay_shift 0 and 8 are the two ends of the tape alphabet)."""
    from mat_mul_b200.env import DemoStore

    N, R, dim_t = 3, 8, 2
    bound = 32767 - R * 8 ** 3 + over
    rng = np.random.default_rng(S + 10 * replay_shift + over)
    hi = 8 if replay_shift == 0 else 0  # the token whose coefficient is +-8
    tok = np.where(rng.random((N, R, 3 * S)) < 0.5, hi, replay_shift).astype(np.int64)
    tok[0] = hi
    sign = np.where((np.arange(S) % 2) == 0, 1, -1)  # neighbouring k: opposite signs
    tgt = (bound * sign[None, None, None, :] * np.where(rng.random((N, S, S, 1)) < 0.5, 1, -1)).astype(np.int64)
    _, gp, tp = geo(S)
    rp = geo(S)[0]
    t16 = np.zeros((N, gp), dtype=np.int16)
    t16[:, :S * rp].reshape(N, S, rp)[:, :, :S * S] = tgt.reshape(N, S, S * S)
    rec = np.zeros((N, R, tp), dtype=np.uint8)
    rec[:, :, :3 * S] = tok
    store = DemoStore(dev(rec), dev(t16), S, replay_shift, target_bound=bound)
    idx = np.concatenate([np.arange(0, N * R, R), np.arange(R - 1, N * R, R), rng.integers(0, N * R, 7)])
    want = sample_reference(tok, tgt, S, dim_t, idx, replay_shift)
    assert np.abs(want).max() == bound + (R - 1) * 8 ** 3  # target +- bound moved away from 0 by R - 1 actions
    st, _, _, _ = store.samples(dev(idx), dim_t, replay_shift=replay_shift)
    assert np.array_equal(st.cpu().numpy(), want.astype(np.float32))


# ---------------------------------------------------------------- K3 tg_demo_accumulate_i16
def greedy_terms(target, shift, S):
    """Token records (R, 3S) with v = e_0 (coefficient 1), u = +-e_0 and w_0 coefficients summing to target."""
    sgn = 1 if target >= 0 else -1
    cmax = 255 - shift
    n = max(1, -(-abs(target) // cmax))
    tok = np.full((n, 3 * S), shift, dtype=np.int64)
    tok[:, 0], tok[:, S] = shift + sgn, shift + 1
    left = abs(target)
    for r in range(n):
        c = min(cmax, left)
        tok[r, 2 * S] = shift + c
        left -= c
    return tok


@pytest.mark.parametrize("S", SIZES)
@pytest.mark.parametrize("shift", [0, 1, 127])
def test_accumulate_i16_int16_edges(env, S, shift):
    targets = [32767, 32768, 0, 1] + ([-32768, -32769, -1] if shift else [])  # shift 0 has no negative coefficient
    recs = [greedy_terms(t, shift, S) for t in targets]
    R = max(len(r) for r in recs)
    tok = np.stack([np.vstack([r, np.full((R - len(r), 3 * S), shift)]) for r in recs])
    want = rank1_sum(tok, shift)
    assert [want[g, 0, 0, 0] for g in range(len(targets))] == targets
    slab16, flags = env.accumulate_demos16(dev(tokens_to_tape3(tok)), S, shift)
    fits = ~((want < -32768) | (want > 32767)).reshape(len(targets), -1).any(axis=1)
    flags = flags.cpu().numpy()
    assert np.array_equal((flags & RANGE) == 0, fits)
    got = dense16(slab16, S)
    assert np.array_equal(got[fits], want[fits])


@pytest.mark.parametrize("S", SIZES)
@pytest.mark.parametrize("shift,tokval", [(0, 128), (127, 255)])
def test_accumulate_i16_does_not_wrap_at_2_pow_32(env, S, shift, tokval):
    # 2048 records of u0 = v0 = w0 = 128: entry (0,0,0) is exactly 2^32, which an int32 sum wraps to 0
    R = 2048
    tok = np.full((2, R, 3 * S), shift, dtype=np.int64)
    tok[0, :, [0, S, 2 * S]] = tokval
    tok[1, :3, 1] = shift + 1  # a sibling that fits: entry (1,0,0) = 3
    tok[1, :3, S] = tok[1, :3, 2 * S] = shift + 1
    slab16, flags = env.accumulate_demos16(dev(tokens_to_tape3(tok)), S, shift)
    flags = flags.cpu().numpy()
    assert flags[0] & RANGE and not flags[1] & RANGE
    assert np.array_equal(dense16(slab16, S)[1], rank1_sum(tok[1:], shift)[0])


@pytest.mark.parametrize("S", [4, 9])
@pytest.mark.parametrize("R", [129, 130])
def test_accumulate_i16_at_the_int32_handover(env, S, R):
    # shift 0, token 255: R * 255^3 passes 2^31 first at R = 130; random tapes on both sides, exact where they fit
    rng = np.random.default_rng(R)
    tok = rng.choice([0, 1, 254, 255], size=(5, R, 3 * S)).astype(np.int64)
    tok[0, :, :] = 1
    tok[0, :, 2 * S] = 32767 // R  # entries R * (32767 // R) <= 32767 and R: the game fits int16
    want = rank1_sum(tok, 0)
    slab16, flags = env.accumulate_demos16(dev(tokens_to_tape3(tok)), S, 0)
    fits = ~((want < -32768) | (want > 32767)).reshape(5, -1).any(axis=1)
    assert np.array_equal((flags.cpu().numpy() & RANGE) == 0, fits)
    assert np.array_equal(dense16(slab16, S)[fits], want[fits])


# ---------------------------------------------------------------- K5 change of basis
@pytest.mark.parametrize("S", [4, 9, 16])
@pytest.mark.parametrize("out_dtype", [torch.int8, torch.int16])
@pytest.mark.parametrize("per_game", [True, False])
def test_change_of_basis_int32_wrap_is_flagged(env, S, out_dtype, per_game):
    """Every entry of T' is 2^32: an int32 accumulator holds 0, which fits int8 and int16."""
    T, A, Bm, Cm = basis_counterexample(S)
    mats = np.stack([A, Bm, Cm]).astype(np.int8)
    rng = np.random.default_rng(S)
    T2 = rng.integers(-2, 3, size=(S, S, S))
    games = np.stack([T, T2, T])
    if per_game:
        eye = np.stack([np.eye(S, dtype=np.int8)] * 3)
        m = np.stack([mats, eye, mats])
        want = np.stack([change_of_basis_ref(T, A, Bm, Cm), T2, change_of_basis_ref(T, A, Bm, Cm)])
    else:
        m = mats[None]
        want = np.stack([change_of_basis_ref(g, A, Bm, Cm) for g in games])
    out, flags = env.change_of_basis(dev(dense_to_slab(games)), dev(m), S, out_dtype=out_dtype)
    flags = flags.cpu().numpy()
    lim = 63 if out_dtype == torch.int8 else 32767
    fits = ~((want < -lim - 1) | (want > lim)).reshape(3, -1).any(axis=1)
    assert np.array_equal((flags & RANGE) == 0, fits), flags
    assert not fits[0] and not fits[2]
    got = slab_to_dense(out.cpu().numpy(), S) if out_dtype == torch.int8 else dense16(out, S)
    assert np.array_equal(got[fits], want[fits])
    if S in (9, 16):  # the f16 and byte-plane guards reject these matrices: the exact kernel computes the game
        assert flags[0] & PATH_EXACT and flags[2] & PATH_EXACT


@pytest.mark.parametrize("out_dtype", [torch.int8, torch.int16])
def test_change_of_basis_4_large_matrices_at_the_edges(env, out_dtype):
    """4x4x4 games whose a-priori bound 128 nA nB nC passes 2^31 (n = largest absolute row sum) while T' cancels to 0,
    or lands exactly on the output's limits and one past them."""
    S = 4
    lim = 63 if out_dtype == torch.int8 else 32767
    big = np.full((S, S), -128, dtype=np.int64)
    e = np.full((S, S), -128, dtype=np.int64)
    e[:, 0] = 1  # A, B: T'[i,j,k] = sum_c C[k,c] T[0,0,c] for a game whose only non-zero entries are T[0,0,.]
    Cm = np.full((S, S), 127, dtype=np.int64)
    Cm[:, 0] = 1  # T' = T[0,0,0] + 127 (T[0,0,1] + T[0,0,2] + T[0,0,3]); nA nB nC = 385^2 382
    cases = [(np.zeros((S, S, S), dtype=np.int64), big, big, big)]
    T = np.zeros((S, S, S), dtype=np.int64)
    T[0, 0, 0], T[1, 0, 0] = 1, -1
    cases.append((T, big, big, big))  # two rows of A that are equal: T' = 0
    for t in (lim, lim + 1, -lim - 1, -lim - 2, 0):
        q, r = divmod(t, 127)
        T = np.zeros((S, S, S), dtype=np.int64)
        T[0, 0, 0] = r
        for c in (1, 2, 3):
            T[0, 0, c] = max(-128, min(127, q))
            q -= T[0, 0, c]
        assert q == 0
        cases.append((T, e, e, Cm))
    games = np.stack([c[0] for c in cases])
    m = np.stack([np.stack(c[1:]) for c in cases])
    want = np.stack([change_of_basis_ref(*c) for c in cases])
    assert [want[g, 0, 0, 0] for g in range(2, 7)] == [lim, lim + 1, -lim - 1, -lim - 2, 0]
    out, flags = env.change_of_basis(dev(dense_to_slab(games)), dev(m.astype(np.int8)), S, out_dtype=out_dtype)
    flags = flags.cpu().numpy()
    fits = ~((want < -lim - 1) | (want > lim)).reshape(len(cases), -1).any(axis=1)
    assert list(fits) == [True, True, True, False, True, False, True]
    assert np.array_equal((flags & RANGE) == 0, fits), flags
    got = slab_to_dense(out.cpu().numpy(), S) if out_dtype == torch.int8 else dense16(out, S)
    assert np.array_equal(got[fits], want[fits])
    # where a game is flagged its entries are still the exact values' low bytes (int8) or halves (int16)
    mask = 0xFF if out_dtype == torch.int8 else 0xFFFF
    assert np.array_equal(got & mask, want & mask)


# ---------------------------------------------------------------- K6 tg_slice_rank
@pytest.mark.parametrize("S", SIZES)
def test_slice_rank_det_equals_p(env, S):
    """A slice with det = 2^31 - 1 (rank 4 over Q, 3 mod 2^31 - 1), one of floor(S/4) such blocks (rank 4 floor(S/4);
    a single prime sees one less per block), and int8 slices across the full range against Python-integer ranks."""
    rng = np.random.default_rng(S)
    B = 4
    T = np.zeros((B, S, S, S), dtype=np.int64)
    T[0, 0, :4, :4] = DET_P
    T[1, S - 1] = block_diag_det_p(S)
    T[2] = rng.integers(-128, 128, size=(S, S, S))
    T[2, 1, :, 3] = 2 * T[2, 1, :, 1] // 2  # a repeated column
    T[3] = rng.integers(-3, 4, size=(S, S, S)) * (rng.random((S, S, S)) < 0.3)
    want = slice_ranks(T)
    assert want[0] == 4 and want[1] == 4 * (S // 4)
    got = env.slice_rank(dev(dense_to_slab(T)), S).cpu().numpy()
    assert np.array_equal(got, want)


# ---------------------------------------------------------------- boundary conversions
@pytest.mark.parametrize("S", SIZES)
def test_pack_f32_edges(env, S):
    from mat_mul_b200.env import _call, _p

    cases = [(-128.0, False), (127.0, False), (-0.0, False), (127.5, True), (128.0, True), (-129.0, True),
             (float("nan"), True), (float("inf"), True), (float("-inf"), True), (-128.5, True)]
    _, gp, _ = geo(S)
    for v, bad in cases:
        heads = torch.zeros((2, S, S, S), dtype=torch.float32, device="cuda")
        heads[1, S - 1, S - 1, S - 1] = v
        heads[0, 0, 0, 0] = -128.0
        slab = torch.empty((2, gp), dtype=torch.int8, device="cuda")
        flag = torch.zeros(1, dtype=torch.int32, device="cuda")
        _call("tg_pack_f32", (heads, slab, flag), _p(heads), S ** 3, _p(slab), 2, S, _p(flag))
        assert bool(flag.item()) == bad, v
        if not bad:
            d = slab_to_dense(slab.cpu().numpy(), S)
            assert d[1, S - 1, S - 1, S - 1] == int(v) and d[0, 0, 0, 0] == -128
    for v, bad in [(-32768.0, False), (32767.0, False), (32768.0, True), (-32769.0, True), (-0.0, False),
                   (0.5, True), (float("nan"), True), (float("inf"), True), (float("-inf"), True)]:
        heads = torch.zeros((1, S, S, S), dtype=torch.float32, device="cuda")
        heads[0, S - 1, 0, S - 1] = v
        slab16 = torch.empty((1, gp), dtype=torch.int16, device="cuda")
        flag = torch.zeros(1, dtype=torch.int32, device="cuda")
        _call("tg_pack_f32_i16", (heads, slab16, flag), _p(heads), S ** 3, _p(slab16), 1, S, _p(flag))
        assert bool(flag.item()) == bad, v
        if not bad:
            assert dense16(slab16, S)[0, S - 1, 0, S - 1] == int(v)


@pytest.mark.parametrize("S", SIZES)
def test_pack_actions_edges(env, S):
    from mat_mul_b200.env import _call, _p

    _, _, tp = geo(S)
    for v, bad in [(0, False), (255, False), (128, False), (-1, True), (256, True), (-128, True), (2**40, True)]:
        a = torch.zeros((2, 3 * S), dtype=torch.int64, device="cuda")
        a[1, 3 * S - 1] = v
        a[0, 0] = 255
        tape = torch.empty((2, tp), dtype=torch.uint8, device="cuda")
        flag = torch.zeros(1, dtype=torch.int32, device="cuda")
        _call("tg_pack_actions_i64", (a, tape, flag), _p(a), _p(tape), 2, S, _p(flag))
        assert bool(flag.item()) == bad, v
        t = tape.cpu().numpy()
        if not bad:
            assert t[1, 3 * S - 1] == v and t[0, 0] == 255
        assert not t[:, 3 * S:].any()
