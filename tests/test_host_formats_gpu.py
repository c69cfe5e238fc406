"""The host-buffer path for int16 and bit slabs on a B200: tg_step_host_i16, tg_rollout_host_i16, tg_step_host_gf2,
tg_rollout_host_gf2 and tg_demo_gen_host_gf2 at 4, 9, 16 and 25, byte for byte against their device twins on the whole
batch (tg_step_i16, tg_rollout_i16, tg_step_gf2, tg_rollout_gf2, tg_demo_gen_gf2).

Contexts of 7 and 64 games per chunk take batches of 1, one chunk, 4 chunks + 1 and 9 chunks + 3 games, so the four
staging buffers wrap more than once and the last chunk is partial.  Host buffers are pinned, pageable, one element off a
16-byte boundary, or the same buffer for input and output (in place)."""
import numpy as np
import pytest
import torch

from mat_mul_b200 import _lib, env
from mat_mul_b200.env import TensorGameError, _p
from tests import gf2_ref, i16_ref
from tests.helpers import dense_to_slab, geo

pytestmark = pytest.mark.gpu

SIZES = (4, 9, 16, 25)
FORMATS = ("i16", "gf2")
DEV = "cuda"
SHIFT = 2
E_ARG = -1
V5, P5 = (-2, -1, 0, 1, 2), (0.05, 0.10, 0.70, 0.10, 0.05)
SIX = ((-3, -2, -1, 0, 1, 2), (0.1, 0.2, 0.15, 0.3, 0.15, 0.1))  # six values: contract v1 at every size
# contract v1, 4 % odd entries: with max_tries = 1 most terms have a factor without an odd entry and are forced
MOSTLY_EVEN = ((-4, -2, -1, 0, 1, 2, 4), (0.2, 0.2, 0.02, 0.2, 0.02, 0.16, 0.2))


def _batches(chunk):
    return (1, chunk, 4 * chunk + 1, 9 * chunk + 3)


def _slab(fmt, S, B, rng, scale=3000):
    """a CPU slab of B games: int16 (B, GP) with entries up to +-scale, or an int32 bit slab (B, GB/4)"""
    T = rng.integers(-scale, scale + 1, size=(B, S, S, S)) * (rng.random((B, S, S, S)) < 0.4)
    if fmt == "i16":
        return torch.from_numpy(i16_ref.dense_to_slab16(T))
    return torch.from_numpy(gf2_ref.dense_to_bits(T))


def _records(fmt, S, shape, rng):
    """uint8 records (*shape, TP): int16 tokens mostly in [0, 2 SHIFT] (some break the bound and raise RANGE), any byte
    for bit slabs"""
    tok = rng.integers(0, 256, size=shape + (3 * S,))
    if fmt == "i16":
        tok = np.where(rng.random(shape + (3 * S,)) < 0.995, rng.integers(0, 2 * SHIFT + 1, size=tok.shape), tok)
    out = np.zeros(shape + (geo(S)[2],), dtype=np.uint8)
    out[..., : 3 * S] = tok
    return torch.from_numpy(out)


def _host(t, mode):
    """a CPU copy of t: pinned, pageable, or pageable one element past a 16-byte boundary"""
    if mode == "pinned":
        return t.clone().pin_memory()
    if mode == "offset":
        buf = torch.empty(t.numel() + 1, dtype=t.dtype)
        assert buf.data_ptr() % 16 == 0
        v = buf[1:].view(t.shape)
        v.copy_(t)
        return v
    return t.clone()


def _empty(shape, dtype, mode):
    return _host(torch.full(shape, 0x55, dtype=dtype), mode)


def _step_host(hs, slab, tape, mode):
    B = slab.shape[0]
    out = slab if mode == "inplace" else _empty(slab.shape, slab.dtype, mode)
    fl, nz = _empty((B,), torch.uint8, mode), _empty((B,), torch.int32, mode)
    hs.step(slab, tape, out, fl, nz, SHIFT)
    return out, fl, nz


def _rollout_host(hs, slab, tape, mode, shift=SHIFT):
    B = slab.shape[0]
    out = slab if mode == "inplace" else _empty(slab.shape, slab.dtype, mode)
    fl, nz, st = _empty((B,), torch.uint8, mode), _empty((B,), torch.int32, mode), _empty((B,), torch.int32, mode)
    hs.rollout(slab, tape, out, fl, nz, st, shift)
    return out, fl, nz, st


def _same(host, device):
    assert len(host) == len(device)
    for h, d in zip(host, device):
        assert torch.equal(h, d.cpu())


MODES = ("pinned", "pageable", "offset", "inplace")


@pytest.mark.parametrize("chunk", (7, 64))
@pytest.mark.parametrize("fmt", FORMATS)
@pytest.mark.parametrize("S", SIZES)
def test_step_and_rollout_match_device_twins(S, fmt, chunk):
    rng = np.random.default_rng(S * 1000 + chunk + (fmt == "gf2"))
    hs = env.HostStepper(S, 0, chunk=chunk)
    try:
        for B in _batches(chunk):
            slab, rec, tape = _slab(fmt, S, B, rng), _records(fmt, S, (B,), rng), _records(fmt, S, (3, B), rng)
            want_step = env.step_batch(slab.to(DEV), rec.to(DEV), S, SHIFT)
            want_roll = env.rollout(slab.to(DEV), tape.to(DEV), S, SHIFT)
            for mode in MODES:
                h_rec, h_tape = _host(rec, mode), _host(tape, mode)
                _same(_step_host(hs, _host(slab, mode), h_rec, mode), want_step)
                _same(_rollout_host(hs, _host(slab, mode), h_tape, mode), want_roll)
                assert torch.equal(h_rec, rec) and torch.equal(h_tape, tape)  # inputs are only read
    finally:
        hs.close()


@pytest.mark.parametrize("fmt", FORMATS)
@pytest.mark.parametrize("S", SIZES)
def test_rollout_cases(S, fmt):
    """K = 0 and 1, reversed demo tapes (every game solves), games frozen mid-tape, int16 games that leave the zone,
    bit-slab tapes of arbitrary bytes"""
    rng = np.random.default_rng(S + 7 * (fmt == "gf2"))
    chunk, B = 7, 4 * 7 + 3
    hs = env.HostStepper(S, 0, chunk=chunk)

    def check(slab, tape, shift=SHIFT, mode="pinned"):
        want = env.rollout(slab.to(DEV), tape.to(DEV), S, shift)
        got = _rollout_host(hs, _host(slab, mode), _host(tape, mode), mode, shift)
        _same(got, want)
        return got

    try:
        slab = _slab(fmt, S, B, rng)
        for K in (0, 1):
            out, _, _, st = check(slab, _records(fmt, S, (K, B), rng))
            assert not st.any() or K == 1
            if K == 0:
                assert torch.equal(out, slab)
        # demos replayed last action first: every game solves
        R = {4: 7, 9: 23, 16: 49, 25: 60}[S]
        if fmt == "i16":
            tape, _, _ = env.make_synthetic_demos(B, R, S, V5, P5, SHIFT, seed=S, device=DEV)
            targets, _ = env.accumulate_demos16(tape, S, SHIFT)
        else:
            tape, targets, _ = env.make_synthetic_demos_gf2(B, R, S, V5, P5, SHIFT, seed=S, device=DEV)
        rev = tape.flip(0).contiguous().cpu()
        targets = targets.cpu()
        for mode in ("pinned", "inplace"):
            out, fl, _, st = check(targets, rev, mode=mode)
            assert not out.any() and bool((fl & env.FLAG_TERMINAL).all()) and int(st.max()) == R
            assert (st == R).float().mean() > 0.9  # a suffix of terms that cancels solves a game early
        # four more records after the demo: games freeze at the step that solves them and ignore the rest
        extra = torch.cat([rev, _records(fmt, S, (4, B), rng)])
        out, fl, _, st = check(targets, extra)
        assert not out.any() and bool((st <= R).all())
        if fmt == "i16":
            # entries next to the zone's edge and coefficients of +-4: steps cross +-16384 and raise RANGE
            T = rng.choice([-16380, -16000, 0, 16000, 16380], size=(B, S, S, S))
            edge = torch.from_numpy(i16_ref.dense_to_slab16(T))
            tok = np.zeros((6, B, geo(S)[2]), dtype=np.uint8)
            tok[..., : 3 * S] = rng.choice([0, 4, 8], size=(6, B, 3 * S))
            _, fl, _, _ = check(edge, torch.from_numpy(tok), shift=4)
            assert bool((fl & env.FLAG_RANGE).any())
        else:
            check(slab, torch.from_numpy(rng.integers(0, 256, size=(5, B, geo(S)[2]), dtype=np.uint8)))
    finally:
        hs.close()


DEMO_CASES = {  # (values, probs, shift, max_tries)
    "v2": (V5, P5, 2, 64),
    "v1": (*SIX, 3, 64),
    "exhausted": (*MOSTLY_EVEN, 4, 1),
}


@pytest.mark.parametrize("case", sorted(DEMO_CASES))
@pytest.mark.parametrize("S", SIZES)
def test_demo_gen_host_gf2_matches_device(S, case):
    values, probs, shift, max_tries = DEMO_CASES[case]
    N, R, first = 4 * 7 + 3, {4: 7, 9: 23, 16: 49, 25: 100}[S], (1 << 32) - 5
    tp, gw = geo(S)[2], env.layout_gf2(S).game_words
    want = env.make_synthetic_demos_gf2(N, R, S, values, probs, shift, seed=S, first_demo=first, device=DEV, max_tries=max_tries)
    hs = env.HostStepper(S, 0, chunk=7)
    try:
        for mode in ("pinned", "offset"):
            got = (_empty((R, N, tp), torch.uint8, mode), _empty((N, gw), torch.int32, mode), _empty((N,), torch.uint8, mode))
            hs.make_demos(*got, shift, values, probs, seed=S, first_demo=first, max_tries=max_tries)
            _same(got, want)
    finally:
        hs.close()
    fl = want[2].cpu()
    if case == "exhausted":
        assert bool((fl & env.FLAG_EXHAUSTED).any())
    if case == "v2" and S <= 16:
        assert not fl.any()  # contract v2 never sets EXHAUSTED


@pytest.mark.parametrize("S", SIZES)
def test_mixed_formats_on_one_context(S):
    """int8 -> int16 -> bits -> int8 on one context: growing the slab staging for int16 disturbs no other format"""
    rng = np.random.default_rng(40 + S)
    chunk, B = 7, 9 * 7 + 3
    hs = env.HostStepper(S, 0, chunk=chunk)
    try:
        T = rng.integers(-3, 4, size=(B, S, S, S)) * (rng.random((B, S, S, S)) < 0.3)
        s8 = torch.from_numpy(dense_to_slab(T))
        rec8 = _records("i16", S, (B,), rng)
        tape8 = _records("i16", S, (3, B), rng)

        def int8_calls():
            _same(_step_host(hs, _host(s8, "pinned"), rec8, "pinned"), env.step_batch(s8.to(DEV), rec8.to(DEV), S, SHIFT))
            _same(_rollout_host(hs, _host(s8, "pageable"), tape8, "pageable"), env.rollout(s8.to(DEV), tape8.to(DEV), S, SHIFT))
            got = (torch.empty((5, B, geo(S)[2]), dtype=torch.uint8), torch.empty(s8.shape, dtype=torch.int8), torch.empty(B, dtype=torch.uint8))
            hs.make_demos(*got, SHIFT, V5, P5, seed=3, first_demo=11)
            _same(got, env.make_synthetic_demos(B, 5, S, V5, P5, SHIFT, seed=3, first_demo=11, device=DEV))

        int8_calls()
        for fmt in FORMATS:
            slab, rec, tape = _slab(fmt, S, B, rng), _records(fmt, S, (B,), rng), _records(fmt, S, (3, B), rng)
            _same(_step_host(hs, _host(slab, "pinned"), rec, "pinned"), env.step_batch(slab.to(DEV), rec.to(DEV), S, SHIFT))
            _same(_rollout_host(hs, _host(slab, "inplace"), tape, "inplace"), env.rollout(slab.to(DEV), tape.to(DEV), S, SHIFT))
        got = (torch.empty((5, B, geo(S)[2]), dtype=torch.uint8), torch.empty((B, env.layout_gf2(S).game_words), dtype=torch.int32),
               torch.empty(B, dtype=torch.uint8))
        hs.make_demos(*got, SHIFT, V5, P5, seed=3, first_demo=11)
        _same(got, env.make_synthetic_demos_gf2(B, 5, S, V5, P5, SHIFT, seed=3, first_demo=11, device=DEV))
        int8_calls()
    finally:
        hs.close()


def test_refused_calls_leave_host_outputs_untouched():
    """a bad shift, a null pointer or a refused alphabet returns TG_E_ARG before any copy: sentinel-filled outputs stay as
    they were, and the context still works afterwards"""
    S, B, R = 9, 4 * 7 + 3, 5
    L = _lib.lib()
    rng = np.random.default_rng(5)
    hs = env.HostStepper(S, 0, chunk=7)
    ctx = hs._ctx
    try:
        tp = geo(S)[2]
        for fmt in FORMATS:
            sfx = "_" + fmt
            slab, rec, tape = _slab(fmt, S, B, rng).pin_memory(), _records(fmt, S, (B,), rng), _records(fmt, S, (3, B), rng)
            out = torch.full(slab.shape, 0x5A5A, dtype=slab.dtype).pin_memory()
            fl, nz, st = torch.full((B,), 0xA5, dtype=torch.uint8), torch.full((B,), -7, dtype=torch.int32), torch.full((B,), -9, dtype=torch.int32)
            sentinels = [t.clone() for t in (out, fl, nz, st)]
            step, roll = getattr(L, "tg_step_host" + sfx), getattr(L, "tg_rollout_host" + sfx)
            calls = {
                "step shift 0": lambda: step(ctx, _p(slab), _p(rec), _p(out), _p(fl), _p(nz), B, 0),
                "step shift 5": lambda: step(ctx, _p(slab), _p(rec), _p(out), _p(fl), _p(nz), B, 5),
                "step null tape": lambda: step(ctx, _p(slab), None, _p(out), _p(fl), _p(nz), B, SHIFT),
                "step null nnz": lambda: step(ctx, _p(slab), _p(rec), _p(out), _p(fl), None, B, SHIFT),
                "rollout shift 0": lambda: roll(ctx, _p(slab), _p(tape), 3, _p(out), _p(fl), _p(nz), _p(st), B, 0),
                "rollout shift 5": lambda: roll(ctx, _p(slab), _p(tape), 3, _p(out), _p(fl), _p(nz), _p(st), B, 5),
                "rollout null steps": lambda: roll(ctx, _p(slab), _p(tape), 3, _p(out), _p(fl), _p(nz), None, B, SHIFT),
                "rollout null in": lambda: roll(ctx, None, _p(tape), 3, _p(out), _p(fl), _p(nz), _p(st), B, SHIFT),
            }
            for label, call in calls.items():
                assert call() == E_ARG, (fmt, label)
                assert all(torch.equal(a, b) for a, b in zip((out, fl, nz, st), sentinels)), (fmt, label)
        h_tape = torch.full((R, B, tp), 0x33, dtype=torch.uint8).pin_memory()
        h_bits = torch.full((B, env.layout_gf2(S).game_words), 0x5A5A, dtype=torch.int32)
        h_fl = torch.full((B,), 0xA5, dtype=torch.uint8)
        sentinels = [t.clone() for t in (h_tape, h_bits, h_fl)]
        alphabets = {
            "no odd value": ((-2, 0, 2), (0.2, 0.6, 0.2), 2),
            "negative probability": ((-1, 0, 1), (0.5, -0.1, 0.6), 1),
            "value beyond shift": ((-2, 0, 2, 1), (0.2, 0.4, 0.2, 0.2), 1),
            "shift 0": ((-1, 0, 1), (0.2, 0.6, 0.2), 0),
            "shift 5": ((-1, 0, 1), (0.2, 0.6, 0.2), 5),
        }
        for label, (values, probs, shift) in alphabets.items():
            v, p = np.asarray(values, dtype=np.int8), np.asarray(probs, dtype=np.float64)
            rc = L.tg_demo_gen_host_gf2(ctx, 1, 0, B, R, shift, v.ctypes.data, p.ctypes.data, len(v), 64, _p(h_tape), _p(h_bits), _p(h_fl))
            assert rc == E_ARG, label
            assert all(torch.equal(a, b) for a, b in zip((h_tape, h_bits, h_fl), sentinels)), label
        v, p = np.asarray(V5, dtype=np.int8), np.asarray(P5, dtype=np.float64)
        assert L.tg_demo_gen_host_gf2(ctx, 1, 0, B, R, SHIFT, None, p.ctypes.data, 5, 64, _p(h_tape), _p(h_bits), _p(h_fl)) == E_ARG
        assert L.tg_demo_gen_host_gf2(ctx, 1, 0, B, R, SHIFT, v.ctypes.data, p.ctypes.data, 5, 64, _p(h_tape), None, _p(h_fl)) == E_ARG
        assert all(torch.equal(a, b) for a, b in zip((h_tape, h_bits, h_fl), sentinels))
        # the context is intact
        hs.make_demos(h_tape, h_bits, h_fl, SHIFT, V5, P5, seed=1)
        _same((h_tape, h_bits, h_fl), env.make_synthetic_demos_gf2(B, R, S, V5, P5, SHIFT, seed=1, device=DEV))
    finally:
        hs.close()


def test_host_stepper_dispatches_on_dtype_and_checks_shapes():
    S, B = 9, 10
    rng = np.random.default_rng(2)
    gp, tp, gw = geo(S)[1], geo(S)[2], env.layout_gf2(S).game_words
    hs = env.HostStepper(S, 0, chunk=4)
    try:
        fl, nz, st = torch.empty(B, dtype=torch.uint8), torch.empty(B, dtype=torch.int32), torch.empty(B, dtype=torch.int32)
        rec, tape = _records("gf2", S, (B,), rng), _records("gf2", S, (2, B), rng)
        for fmt, dtype, width in (("i16", torch.int16, gp), ("gf2", torch.int32, gw)):
            slab = _slab(fmt, S, B, rng)
            out = torch.empty_like(slab)
            hs.step(slab, rec if fmt == "gf2" else _records("i16", S, (B,), rng), out, fl, nz, SHIFT)
            assert out.dtype == dtype and out.shape == (B, width)
            bad = [(torch.zeros((B, width + 4), dtype=dtype), out),   # slab of the wrong width
                   (slab, torch.empty((B, width), dtype=torch.int8 if fmt == "gf2" else torch.int32)),  # out of another dtype
                   (slab, torch.empty((B - 1, width), dtype=dtype))]  # out of another batch
            for s_, o_ in bad:
                with pytest.raises(TensorGameError):
                    hs.step(s_, rec, o_, fl, nz, SHIFT)
                with pytest.raises(TensorGameError):
                    hs.rollout(s_, tape, o_, fl, nz, st, SHIFT)
            with pytest.raises(TensorGameError):
                hs.step(slab, tape, out, fl, nz, SHIFT)  # a K-step tape for one step
            with pytest.raises(TensorGameError):
                hs.rollout(slab, rec, out, fl, nz, st, SHIFT)  # one record per game for a rollout
            with pytest.raises(TensorGameError):
                hs.rollout(slab, tape, out, fl, nz[:-1].contiguous(), st, SHIFT)
        demo_tape = torch.empty((3, B, tp), dtype=torch.uint8)
        with pytest.raises(TensorGameError):
            hs.make_demos(demo_tape, torch.empty((B, gp), dtype=torch.int16), fl, SHIFT, V5, P5)
        with pytest.raises(TensorGameError):
            hs.make_demos(demo_tape, torch.empty((B, gw + 1), dtype=torch.int32), fl, SHIFT, V5, P5)
        hs.make_demos(demo_tape, torch.empty((B, gw), dtype=torch.int32), fl, SHIFT, V5, P5)
    finally:
        hs.close()
