"""25x25x25 (5x5 matrix multiplication) on the game path: every entry point bit for bit against the CPU oracle."""
import numpy as np
import pytest
import torch

from oracle import tg_oracle as orc
from tests import oracle_any_s as orx
from tests.helpers import dense_to_slab, geo, slab_to_dense, tape3_to_tokens, tokens_to_tape, tokens_to_tape3

pytestmark = pytest.mark.gpu

S = 25
RP, GP, TP = geo(S)
V3, P3 = (-1, 0, 1), (0.15, 0.7, 0.15)
V5, P5 = (-2, -1, 0, 1, 2), (0.05, 0.10, 0.70, 0.10, 0.05)
DEV = "cuda"


@pytest.fixture(scope="module")
def env():
    from mat_mul_b200 import env as e

    assert torch.cuda.is_available()
    return e


def rank1(tok, shift):
    u, v, w = (np.asarray(tok[m * S:(m + 1) * S], dtype=np.int64) - shift for m in range(3))
    return np.einsum("i,j,k->ijk", u, v, w)


def to_dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def dense16(slab16):
    return slab16.cpu().numpy()[:, : S * RP].reshape(-1, S, RP)[:, :, : S * S].reshape(-1, S, S, S).astype(np.int32)


@pytest.fixture(scope="module")
def demos():
    """Reference-style demos (values -1/0/1, R ~ 100) from the throughput sampler, with the oracle's tokens and targets."""
    N, R, shift = 24, 100, 1
    tok, tgt, ex = orx.demos_philox(9, 3, N, V3, P3, R, S, shift)
    return N, R, shift, tok, tgt, ex


def test_layout(env):
    lay = env.layout(S)
    assert (lay.row_pitch, lay.game_pitch, lay.token_pitch) == (628, 15712, 80)


def test_boundary_conversions_every_alignment(env):
    rng = np.random.default_rng(1)
    B = 5
    T = rng.integers(-128, 128, size=(B, S, S, S)).astype(np.int32)
    slab = env.pack_states(to_dev(T.astype(np.float32)), S)
    assert np.array_equal(slab_to_dense(slab.cpu().numpy(), S), T)
    n = S ** 3
    for off in range(4):  # games at every 4-byte alignment of a float buffer, bytes around them untouched
        buf = torch.full((B * n + 8,), -7.0, device=DEV)
        out = buf[off: off + B * n].view(B, S, S, S)
        env.expand_states(slab, S, out=out)
        torch.cuda.synchronize()
        host = buf.cpu().numpy()
        assert np.array_equal(host[off: off + B * n].reshape(B, S, S, S), T) and (host[:off] == -7).all() and (host[off + B * n:] == -7).all()
        assert torch.equal(env.pack_states(out, S), slab)
    T16 = rng.integers(-32768, 32768, size=(B, S, S, S)).astype(np.int32)
    s16 = env.pack_states16(to_dev(T16.astype(np.float32)), S)
    assert np.array_equal(dense16(s16), T16) and np.array_equal(env.expand_states16(s16, S).cpu().numpy(), T16)
    acts = rng.integers(0, 9, size=(B, 3 * S))
    tape = env.pack_actions(to_dev(acts), S)
    assert np.array_equal(tape.cpu().numpy(), tokens_to_tape(acts)) and np.array_equal(env.unpack_actions(tape, S).cpu().numpy(), acts)
    with pytest.raises(env.TensorGameError):
        env.pack_states(to_dev(np.full((1, S, S, S), 200.0, dtype=np.float32)), S)


@pytest.mark.parametrize("B", [1, 3, 257, 5000])
def test_step(env, B):
    rng = np.random.default_rng(B)
    for shift in (1, 2, 3, 4):
        T = rng.integers(-63, 64, size=(B, S, S, S)).astype(np.int32)  # results stay inside int8: exact
        tok = rng.integers(0, 2 * shift + 1, size=(B, 3 * S)).astype(np.int32)
        tok[0, S: 2 * S] = shift  # null action
        if B > 2:
            T[1] = rank1(tok[1], shift)  # solved by its action
            tok[2, 5] = 2 * shift + 1  # breaks the token bound: RANGE
        want, wf, wn = orc.step_batch(T, tok, shift)
        slab, tape = to_dev(dense_to_slab(T)), to_dev(tokens_to_tape(tok))
        out, flags, nnz = env.step_batch(slab, tape, S, shift)
        fl = flags.cpu().numpy()
        ok = np.ones(B, dtype=bool)
        if B > 2:
            ok[2] = False
            assert fl[2] & 4 and fl[1] & 1
        assert np.array_equal(slab_to_dense(out.cpu().numpy(), S)[ok], want[ok])
        assert np.array_equal(fl[ok] & 3, wf[ok] & 3) and np.array_equal(nnz.cpu().numpy()[ok], wn[ok])
        assert fl[0] & 2
        env.step_batch(slab, tape, S, shift, out=slab)  # in place
        assert torch.equal(slab, out)


def test_demo_replay_reaches_zero(env, demos):
    N, R, shift, tok, tgt, _ = demos
    tape, slab, fl = env.make_synthetic_demos(N, R, S, V3, P3, shift, seed=9, first_demo=3, device=DEV)
    cur = slab
    for r in reversed(range(R)):
        cur, flags, nnz = env.step_batch(cur, tape[r].contiguous(), S, shift)
    assert not cur.any() and bool((flags & 1).all()) and not nnz.any()


def test_expand_children(env, demos):
    N, R, shift, tok, tgt, _ = demos
    k = 6
    tape = to_dev(tokens_to_tape3(tok[:, :k])).permute(1, 0, 2).contiguous()
    parents = tgt.copy()
    parents[0] = rank1(tok[0, 2], shift)  # child 2 of parent 0 solves it
    kids, kf, kn, kk = env.expand_children(to_dev(dense_to_slab(parents)), tape, S, shift)
    for c in range(k):
        want, wf, wn = orc.step_batch(parents, tok[:, c], shift)
        assert np.array_equal(slab_to_dense(kids[:, c].contiguous().cpu().numpy(), S), want)
        assert np.array_equal(kf[:, c].cpu().numpy() & 3, wf) and np.array_equal(kn[:, c].cpu().numpy(), wn)
        assert np.array_equal(kk[:, c].cpu().numpy().view(np.uint64), orc.state_key_batch(want))
    assert kf[0, 2].item() & 1 and kk[0, 2].item() == 0


@pytest.mark.parametrize("B,K", [(1, 0), (3, 4), (5, 8), (7, 9), (300, 23)])
def test_rollout_replay(env, B, K):
    rng = np.random.default_rng(K)
    shift = 2
    tape = rng.integers(0, 2 * shift + 1, size=(B, K, 3 * S)).astype(np.int32) * (rng.random((B, K, 3 * S)) < 0.3)
    tape = (tape + shift * (tape == 0)).astype(np.int32)
    T = rng.integers(-3, 4, size=(B, S, S, S)).astype(np.int32)
    if K >= 4:
        T[0] = sum(rank1(tape[0, t], shift) for t in range(K // 2))  # solved in the middle of the tape
    slab, tp = to_dev(dense_to_slab(T)), to_dev(tokens_to_tape3(tape))
    out, fl, nz, st = env.rollout(slab, tp, S, shift)
    wo, wf, wn, ws = orx.rollout_batch(T, tape, shift)
    assert np.array_equal(slab_to_dense(out.cpu().numpy(), S), wo) and np.array_equal(st.cpu().numpy(), ws)
    assert np.array_equal(fl.cpu().numpy() & 1, wf & 1) and np.array_equal(nz.cpu().numpy(), wn)
    if K >= 4:
        assert st[0].item() == K // 2 and not out[0].any()
    r_out, r_fl, r_nz = env.replay(slab, tp, S, shift)
    want = np.stack([T[b].astype(np.int64) - sum((rank1(tape[b, t], shift) for t in range(K)), np.zeros((S, S, S), np.int64)) for b in range(B)])
    assert np.array_equal(slab_to_dense(r_out.cpu().numpy(), S), want)


def test_state_key_and_slice_rank(env, demos):
    N, R, shift, tok, tgt, _ = demos
    T = np.concatenate([np.zeros((1, S, S, S), np.int32), orc.build_matmul_tensor(5)[None], tgt]).astype(np.int32)
    T = np.clip(T, -64, 63)
    keys = env.state_keys(to_dev(dense_to_slab(T)), S).cpu().numpy().view(np.uint64)
    assert keys[0] == 0 and np.array_equal(keys, orc.state_key_batch(T))
    a, b = np.clip(T[2], -30, 30), np.clip(T[3], -30, 30)
    kab = env.state_keys(to_dev(dense_to_slab(np.stack([a, b, a + b]))), S).cpu().numpy().view(np.uint64)
    assert kab[2] == (int(kab[0]) + int(kab[1])) % 2 ** 64  # linear in the state
    ranks = env.slice_rank(to_dev(dense_to_slab(T)), S).cpu().numpy()
    assert np.array_equal(ranks, orc.slice_rank_batch(T)) and ranks[1] == 125 and ranks[0] == 0


@pytest.mark.parametrize("values,probs,shift,max_tries", [(V3, P3, 1, 64), (V5, P5, 2, 64), ((-1, 0, 1), (0.001, 0.998, 0.001), 1, 2),
                                                          ((-3, -1, 0, 1, 2, 3), (0.1, 0.1, 0.4, 0.2, 0.1, 0.1), 3, 64)])
def test_demo_gen_and_accumulate(env, values, probs, shift, max_tries):
    N, R = 40, 30
    tok, tgt, ex = orx.demos_philox(5, 11, N, values, probs, R, S, shift, max_tries=max_tries)
    tape, slab, fl = env.make_synthetic_demos(N, R, S, values, probs, shift, seed=5, first_demo=11, max_tries=max_tries, device=DEV)
    assert np.array_equal(tape3_to_tokens(tape.cpu().numpy(), S), tok)
    fl = fl.cpu().numpy()
    fits = ((tgt >= -64) & (tgt <= 63)).reshape(N, -1).all(1)
    assert np.array_equal((fl & 4) == 0, fits)
    assert np.array_equal(slab_to_dense(slab.cpu().numpy(), S)[fits], tgt[fits])
    assert np.array_equal(slab.cpu().numpy().view(np.uint8)[:, : S * RP].reshape(N, S, RP)[:, :, : S * S].reshape(N, S, S, S),
                          (tgt & 0xFF).astype(np.uint8))  # entries modulo 256
    assert ((fl & 8) != 0).sum() > 0 if ex else not (fl & 8).any()
    s2, f2 = env.accumulate_demos(tape, S, shift)
    assert torch.equal(s2, slab) and np.array_equal(f2.cpu().numpy(), fl & 4)
    s16, f16 = env.accumulate_demos16(tape, S, shift)
    assert np.array_equal(dense16(s16), tgt) and not f16.any()


def test_accumulate_beyond_int8(env):
    R, N, shift = 60, 6, 4
    tok = np.full((N, R, 3 * S), 8, dtype=np.int32)  # every coefficient +4: entries 60 * 64 = 3840
    tok[1, :, 3] = 0
    tape = to_dev(tokens_to_tape3(tok))
    want = np.stack([sum(rank1(tok[n, r], shift) for r in range(R)) for n in range(N)])
    s16, f16 = env.accumulate_demos16(tape, S, shift)
    assert np.array_equal(dense16(s16), want) and not f16.any()
    s8, f8 = env.accumulate_demos(tape, S, shift)
    assert (f8.cpu().numpy() & 4).all()
    assert np.array_equal(s8.cpu().numpy().view(np.uint8)[:, : S * RP].reshape(N, S, RP)[:, :, : S * S].reshape(N, S, S, S),
                          (want & 0xFF).astype(np.uint8))


def test_parity_mode_create_synthetic_demo(env):
    from mat_mul_b200 import utils
    from tests.test_s25_oracle import torch_create_synthetic_demo

    torch.manual_seed(77)
    acts, target = utils.create_synthetic_demo(torch.tensor(V3), torch.tensor(P3), 5, S, 1)
    after = torch.rand(4, dtype=torch.float64)
    torch.manual_seed(77)
    want_acts, want_tgt = torch_create_synthetic_demo(V3, P3, 5, 1)
    assert torch.equal(torch.stack(acts), want_acts) and torch.equal(target, want_tgt)
    assert torch.equal(torch.rand(4, dtype=torch.float64), after)
    tok, tgt, used = orx.demos_seeded(3, V5, P5, 7, S, 2, 12)
    tape, slab, _, consumed = env.demos_from_seed(12, 7, S, V5, P5, 2, seed=3, device=DEV)
    assert consumed == used and np.array_equal(tape3_to_tokens(tape.cpu().numpy(), S), tok)
    assert np.array_equal(slab_to_dense(slab.cpu().numpy(), S), tgt)


@pytest.mark.parametrize("dim_t", [1, 2, 4])
@pytest.mark.parametrize("R", [1, 100])
def test_demo_samples(env, dim_t, R):
    N, shift = 6, 1
    tok, tgt, _ = orx.demos_philox(2, 0, N, V3, P3, R, S, shift)
    tape, slab, _ = env.make_synthetic_demos(N, R, S, V3, P3, shift, seed=2, first_demo=0, device=DEV)
    idx_np = np.array([0, N * R - 1, R // 2, N * R + 5, 3 * R + (R - 1) // 3, -1])
    idx = to_dev(idx_np)
    want = np.zeros((len(idx_np), dim_t, S, S, S), dtype=np.float32)
    for b, i in enumerate(idx_np):
        if 0 <= i < N * R:
            want[b] = orx.demo_getitem(tok[i // R], tgt[i // R], dim_t, i % R, replay_shift=shift)[0]
    good = (idx_np >= 0) & (idx_np < N * R)
    st, sc, ac, rw = env.demo_samples(tape, slab, idx[good], S, dim_t, replay_shift=shift)
    assert np.array_equal(st.cpu().numpy(), want[good])
    slab16, _ = env.accumulate_demos16(tape, S, shift)
    for targets in (slab, slab16):
        store = env.DemoStore.from_tape(tape, targets, S, shift)
        st, sc, ac, rw = store.samples(idx, dim_t, replay_shift=shift)
        assert np.array_equal(st.cpu().numpy(), want)
        gi = idx_np[good]
        assert np.array_equal(ac.cpu().numpy()[good], tok.reshape(N * R, -1)[gi])
        assert np.array_equal(sc.cpu().numpy().reshape(-1)[good], (R - gi % R).astype(np.float32))
        assert np.array_equal(rw.cpu().numpy().reshape(-1)[good], -(gi % R + 1).astype(np.float32))
    # states at an unaligned float offset
    from mat_mul_b200 import _lib
    from mat_mul_b200.env import _p, _stream

    store = env.DemoStore.from_tape(tape, slab, S, shift)
    nb = int(good.sum())
    n = dim_t * S ** 3
    buf = torch.full((nb * n + 4,), -5.0, device=DEV)
    sc, rw = torch.empty(nb, device=DEV), torch.empty(nb, device=DEV)
    ac = torch.empty((nb, 3 * S), dtype=torch.int64, device=DEV)
    ig = idx[good].contiguous()
    rc = _lib.lib().tg_demo_sample_dm(_p(store.records), _p(store.targets), 0, 127, N, R, S, dim_t, shift, _p(ig), nb,
                                      buf.data_ptr() + 4, _p(sc), _p(ac), _p(rw), _stream())
    assert rc == 0
    torch.cuda.synchronize()
    host = buf.cpu().numpy()
    assert np.array_equal(host[1: 1 + nb * n].reshape(want[good].shape), want[good]) and host[0] == -5 and (host[1 + nb * n:] == -5).all()


def test_host_paths(env, demos):
    N, R, shift, tok, tgt, _ = demos
    R = 9
    tok, tgt, _ = orx.demos_philox(4, 0, N, V5, P5, R, S, 2)
    tape, slab, _ = env.make_synthetic_demos(N, R, S, V5, P5, 2, seed=4, first_demo=0, device=DEV)
    hs = env.HostStepper(S, 0, chunk=7)
    h_out = torch.empty_like(slab).cpu()
    h_fl, h_nz, h_st = torch.empty(N, dtype=torch.uint8), torch.empty(N, dtype=torch.int32), torch.empty(N, dtype=torch.int32)
    hs.step(slab.cpu(), tape[R - 1].cpu().contiguous(), h_out, h_fl, h_nz, 2)
    d_out, d_fl, d_nz = env.step_batch(slab, tape[R - 1].contiguous(), S, 2)
    assert torch.equal(h_out, d_out.cpu()) and torch.equal(h_fl, d_fl.cpu()) and torch.equal(h_nz, d_nz.cpu())
    hs.rollout(slab.cpu(), tape.flip(0).contiguous().cpu(), h_out, h_fl, h_nz, h_st, 2)
    assert not h_out.any() and bool((h_fl & 1).all())
    h_tape, h_slab = torch.empty((R, N, TP), dtype=torch.uint8), torch.empty((N, GP), dtype=torch.int8)
    hs.make_demos(h_tape, h_slab, h_fl, 2, V5, P5, seed=4, first_demo=0)
    assert torch.equal(h_tape, tape.cpu()) and torch.equal(h_slab, slab.cpu())
    hs.close()


def test_bad_arguments_and_size_limited_entry_points(env):
    from mat_mul_b200 import _lib
    from mat_mul_b200.env import _p, _stream

    L = _lib.lib()
    st = _stream()
    slab = torch.zeros((4, GP + 16), dtype=torch.int8, device=DEV)
    tape = torch.full((4, TP + 16), 1, dtype=torch.uint8, device=DEV)
    out = torch.zeros_like(slab)
    fl, nz = torch.empty(4, dtype=torch.uint8, device=DEV), torch.empty(4, dtype=torch.int32, device=DEV)
    s, t, o = slab.data_ptr(), tape.data_ptr(), out.data_ptr()
    assert L.tg_step(s, t, o, _p(fl), _p(nz), 4, S, 1, st) == 0
    assert L.tg_step(None, t, o, _p(fl), _p(nz), 4, S, 1, st) == -1
    assert L.tg_step(s + 4, t, o, _p(fl), _p(nz), 4, S, 1, st) == -1
    assert L.tg_rollout(s + 4, t, TP, 1, o, _p(fl), _p(nz), _p(nz), 4, S, 1, st) == -1
    assert L.tg_rollout(s, t, TP, 1, o, _p(fl), _p(nz), None, 4, S, 1, st) == -1
    assert L.tg_expand_children(s, t + 8, 1, o, _p(fl), _p(nz), None, 4, S, 1, st) == -1
    assert L.tg_expand_children(s, t, 100000, o, _p(fl), _p(nz), None, 4, S, 1, st) == -1  # tokens overflow shared memory
    assert L.tg_demo_accumulate(t + 8, TP, 4, 1, S, 1, s, _p(fl), st) == -1
    assert L.tg_demo_accumulate_i16(t, TP, 4, 1, S, 1, None, _p(fl), st) == -1
    assert L.tg_pack_f32(None, S ** 3, s, 4, S, None, st) == -1
    assert L.tg_expand_f32(s + 4, None, S ** 3, 4, S, st) == -1
    assert L.tg_slice_rank(None, _p(nz), 4, S, st) == -1 and L.tg_state_key(s, None, 4, S, st) == -1
    assert L.tg_tape_to_demo_major(t + 4, TP, t, 4, 1, S, st) == -1
    assert L.tg_demo_from_ustream_workspace(3 * S * 10, S) > 0
    mats = torch.zeros((4, 3, S, S), dtype=torch.int8, device=DEV)
    # the change of basis and the tensor-core accumulate keep their sizes: 25 is rejected
    assert L.tg_change_of_basis(s, _p(mats), 1, o, _p(fl), 4, S, st) == -1
    assert L.tg_change_of_basis_i16(s, _p(mats), 1, o, _p(fl), 4, S, st) == -1
    assert L.tg_change_of_basis_factors(t, TP, 1, _p(mats), 1, t, TP, 1, _p(fl), 4, 1, S, st) == -1
    assert L.tg_sample_unimodular(1, 0, 4, S, 0.3, _p(mats), st) == -1
    assert L.tg_demo_accumulate_tc(t, TP, 4, 1, S, 1, s, _p(fl), st) == -1
    import ctypes as C

    tabs = np.zeros((8, 128), dtype=np.uint16)
    vals, probs = np.array(V3, dtype=np.int8), np.array(P3, dtype=np.float64)
    assert L.tg_demo_alias_tables(vals.ctypes.data_as(C.c_void_p), probs.ctypes.data_as(C.c_void_p), 3, S,
                                  tabs.ctypes.data_as(C.c_void_p)) == -1  # contract v1 at 25x25x25
    torch.cuda.synchronize()


def test_tensor_game_dataset_and_actor(env, tmp_path, monkeypatch):
    from torch.utils.data import DataLoader

    from mat_mul_b200 import act, datasets
    from tests.fake_model import FakeAlphaTensor

    monkeypatch.chdir(tmp_path)
    np.random.seed(0)
    torch.manual_seed(0)
    ds = datasets.TensorGameDataset(16, 1.0, 6, 2, S, "cpu")
    assert ds.start_tensor.shape == (2, S, S, S) and int(ds.start_tensor[0].sum()) == 125
    st, sc, ac, rw = next(iter(DataLoader(ds, batch_size=8)))
    assert st.shape == (8, 2, S, S, S) and ac.shape == (8, 3 * S) and sc.shape == (8, 1) and rw.shape == (8, 1)
    fm = FakeAlphaTensor(dim_3d=S, n_samples=4, n_logits=3, seed=1)
    init = ds.start_tensor.float()
    state_seq, policy_seq, reward_seq = act.actor_prediction(fm, init, 4, 3, 100)
    assert fm.calls > 0 and len(state_seq) >= 1
    heads = [s.reshape(-1, S, S, S)[0].numpy().astype(np.int32) for s in state_seq]  # slot 0 of each state
    assert np.array_equal(heads[0], orc.build_matmul_tensor(5))
    for a, b in zip(heads, heads[1:]):  # every state is its predecessor minus one rank-1 action
        diff = (a - b).astype(np.float64)
        assert diff.any() and np.linalg.matrix_rank(diff.reshape(S, S * S)) == 1 and np.linalg.matrix_rank(diff.reshape(S * S, S)) == 1
        nz = np.argwhere(diff != 0)[0]
        u, v, w = diff[:, nz[1], nz[2]], diff[nz[0], :, nz[2]], diff[nz[0], nz[1], :]
        tok = np.concatenate([u, v / diff[tuple(nz)], w / diff[tuple(nz)]]).astype(np.int64) + 1
        assert np.array_equal(orc.step_batch(a[None], tok[None], 1)[0][0], b)  # the oracle step of the parent
