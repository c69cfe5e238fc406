"""Rectangular products <n, m, p> on the CPU: the restatement of contract box v1 against contract v1, the embedded
matmul tensors, the naive factorization, box-preserving bases, and the argument rules of tg_demo_gen_box(_gf2)."""
import ctypes as C
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from mat_mul_b200 import env, utils
from oracle import tg_oracle as orc
from tests import box_ref, gf2_demo_ref, oracle_any_s as oas
from tests.basis_inverse_ref import inverses_int8

ROOT = Path(__file__).resolve().parents[1]
OK, E_ARG = 0, -1
V3, P3 = (-1, 0, 1), (0.15, 0.7, 0.15)
V5, P5 = (-2, -1, 0, 1, 2), (0.05, 0.10, 0.70, 0.10, 0.05)
V6, P6 = (-2, -1, 0, 1, 2, 3), (0.05, 0.1, 0.6, 0.1, 0.1, 0.05)


@pytest.mark.parametrize("S", box_ref.SIZES)
@pytest.mark.parametrize("values,probs,shift", [(V3, P3, 1), (V5, P5, 2), (V6, P6, 3)])
def test_full_box_is_contract_v1(S, values, probs, shift):
    tok, tgt, ex = box_ref.demos(11, 5, 24, values, probs, 7, S, shift, (S, S, S), max_tries=3)
    wtok, wtgt, wex = oas.demos_philox_v1(11, 5, 24, values, probs, 7, S, shift, max_tries=3)
    assert np.array_equal(tok, wtok) and np.array_equal(tgt, wtgt) and int(ex.sum()) <= wex
    assert wex == 0 or ex.any()


@pytest.mark.parametrize("S", box_ref.SIZES)
def test_full_box_mod2_is_v1_mod2(S):
    d = (np.uint64(3) + np.repeat(np.arange(16, dtype=np.uint64), 5)).astype(np.uint64)
    r = np.tile(np.arange(5, dtype=np.uint32), 16)
    f, pend = gf2_demo_ref._v1(9, d, r, V6, P6, S, 4)
    tok, tgt, ex = box_ref.demos(9, 3, 16, V6, P6, 5, S, 3, (S, S, S), max_tries=4, gf2=True)
    assert np.array_equal(tok, (f.reshape(16, 5, 3 * S) + 3).astype(np.int32))
    assert np.array_equal(ex, pend.reshape(16, 5).any(1))


@pytest.mark.parametrize("gf2", [False, True])
def test_factors_stay_in_the_box(gf2):
    for n, m, p, S, box in box_ref.shapes()[::7]:
        tok, tgt, ex = box_ref.demos(1, 0, 16, V5, P5, 9, S, 2, box, gf2=gf2)
        f = tok.reshape(16, 9, 3, S).astype(np.int64) - 2
        ins = box_ref.inside(S, box)
        assert not (f * ~ins).any()
        assert ((f % 2 == 1) if gf2 else (f != 0)).any(3).all()
        nu, nv, nw = box
        outside = np.ones((S, S, S), dtype=bool)
        outside[:nu, :nv, :nw] = False
        assert not tgt[:, outside].any()


def test_exhausted_term_is_the_unit_triple():
    tok, tgt, ex = box_ref.demos(2, 0, 8, V3, (0.0001, 0.9998, 0.0001), 3, 9, 1, (2, 3, 6), max_tries=1)
    assert ex.all()
    f = tok.reshape(8, 3, 3, 9) - 1
    want = np.zeros((3, 9), dtype=np.int64)
    want[:, 0] = 1
    assert (f == want).all()


def test_matmul_tensor_contracts_to_the_product():
    rng = np.random.default_rng(0)
    for n, m, p, S, box in box_ref.shapes():
        T = env.matmul_tensor(n, m, p).numpy().astype(np.int64)
        assert env.matmul_box(n, m, p) == (S, box) and T.shape == (S, S, S)
        assert np.array_equal(T, box_ref.matmul_tensor(n, m, p, S))
        A, B = rng.integers(-9, 10, (n, m)), rng.integers(-9, 10, (m, p))
        a, b = np.zeros(S, dtype=np.int64), np.zeros(S, dtype=np.int64)
        a[: n * m], b[: m * p] = A.reshape(-1), B.reshape(-1)
        c = np.einsum("abc,a,b->c", T, a, b)
        assert np.array_equal(c[: n * p], (A @ B).reshape(-1)) and not c[n * p:].any()
        F = box_ref.naive_factors(n, m, p, S)
        assert np.array_equal(np.einsum("ti,tj,tk->ijk", F[:, 0], F[:, 1], F[:, 2]), T)


@pytest.mark.parametrize("n", [1, 2, 3, 4, 5])
def test_square_target_is_the_oracles(n):
    T = env.matmul_tensor(n, n, n, S=n * n if n > 1 else 4).numpy()
    assert np.array_equal(T[: n * n, : n * n, : n * n], orc.build_matmul_tensor(n))
    assert np.array_equal(T[: n * n, : n * n, : n * n], utils.build_matmul_tensor(1, n, n, n)[0].numpy())


def test_matmul_box_refuses_what_does_not_fit():
    for bad in [(1, 6, 5), (6, 5, 1), (3, 3, 9), (0, 2, 2)]:
        with pytest.raises(env.TensorGameError):
            env.matmul_box(*bad)
    with pytest.raises(env.TensorGameError):
        env.matmul_tensor(3, 3, 3, S=4)


@pytest.mark.parametrize("S", [4, 9, 16])
def test_box_bases_are_unimodular_and_keep_the_box(S):
    mats = orc.sample_unimodular(5, 0, 64, S)
    for n, m, p, S2, box in box_ref.shapes():
        if S2 != S:
            continue
        got = env.box_bases(torch.from_numpy(mats.astype(np.int8)), box).numpy().astype(np.int64)
        assert np.array_equal(got, box_ref.box_bases(mats, box))
        inv, fl = inverses_int8(got)
        assert not fl.any()
        T = box_ref.matmul_tensor(n, m, p, S)
        for g in range(0, 64, 16):
            T2 = orc.change_of_basis(T, *got[g])
            nu, nv, nw = box
            outside = np.ones((S, S, S), dtype=bool)
            outside[:nu, :nv, :nw] = False
            assert not T2[outside].any()
            assert np.array_equal(orc.change_of_basis(T2, *inv[g]), T)


def test_box_bases_gf2_blocks():
    S = 9
    rng = np.random.default_rng(1)
    bits = rng.integers(0, 1 << S, (4, 3, S)).astype(np.int32)
    got = env.box_bases(torch.from_numpy(bits), (2, 6, 9)).numpy()
    for f, k in enumerate((2, 6, 9)):
        for r in range(S):
            want = (int(bits[0, f, r]) & ((1 << k) - 1)) if r < k else 1 << r
            assert int(got[0, f, r]) == want


# ---------------------------------------------------------------- argument rules (no device)
def table():
    vals = (C.c_int8 * 3)(-1, 0, 1)
    probs = (C.c_double * 3)(0.15, 0.7, 0.15)
    even = (C.c_int8 * 2)(0, 2)
    neg = (C.c_double * 3)(-0.1, 0.7, 0.4)
    base = 1 << 20
    rows = []

    def row(label, fn, want, S=4, N=1, R=3, box=(1, 1, 1), shift=1, v=vals, p=probs, nv=3, mt=8, tape=base, stride=256,
            tgt=base + 4096):
        args = [C.c_uint64(1), C.c_uint64(0), C.c_int64(N), R, S, *box, shift, C.cast(v, C.c_void_p) if v else None,
                C.cast(p, C.c_void_p) if p else None, nv, mt, C.c_void_p(tape) if tape else None, C.c_int64(stride),
                C.c_void_p(tgt) if tgt else None, None, None]
        rows.append((f"{fn} {label}", fn, args, want))

    for fn in ("tg_demo_gen_box", "tg_demo_gen_box_gf2"):
        for S in box_ref.SIZES:
            for f in range(3):
                for bad in (0, -1, S + 1):
                    box = [1, 1, 1]
                    box[f] = bad
                    row(f"S={S} box[{f}]={bad} empty", fn, E_ARG, S=S, N=0, box=tuple(box), tape=0, tgt=0)
                    row(f"S={S} box[{f}]={bad}", fn, E_ARG, S=S, box=tuple(box))
            row(f"S={S} full box empty batch", fn, OK, S=S, N=0, box=(S, S, S), tape=0, tgt=0, v=None, p=None)
            row(f"S={S} R=0", fn, E_ARG, S=S, R=0)
            row(f"S={S} R=65536", fn, E_ARG, S=S, R=65536)
            row(f"S={S} N<0", fn, E_ARG, S=S, N=-1)
        for S in (-4, 0, 1, 3, 5, 8, 36):
            row(f"S={S}", fn, E_ARG, S=S, N=0)
        for label, kw in [("shift=0", dict(shift=0)), ("shift=5", dict(shift=5)), ("n_values=0", dict(nv=0)),
                          ("n_values=9", dict(nv=9)), ("max_tries=0", dict(mt=0)), ("max_tries=65536", dict(mt=65536)),
                          ("tape NULL", dict(tape=0)), ("target NULL", dict(tgt=0)), ("values NULL", dict(v=None)),
                          ("probs NULL", dict(p=None)), ("tape+8", dict(tape=base + 8)), ("target+4", dict(tgt=base + 4096 + 4)),
                          ("stride 8", dict(stride=8)), ("negative probability", dict(p=neg)),
                          ("value outside shift", dict(shift=1, v=(C.c_int8 * 3)(-2, 0, 1)))]:
            row(label, fn, E_ARG, **kw)
    rows.append(("tg_demo_gen_box_gf2 no odd value", "tg_demo_gen_box_gf2",
                 [C.c_uint64(1), C.c_uint64(0), C.c_int64(1), 3, 4, 1, 1, 1, 2, C.cast(even, C.c_void_p),
                  C.cast(probs, C.c_void_p), 2, 8, C.c_void_p(base), C.c_int64(256), C.c_void_p(base + 4096), None, None], E_ARG))
    return rows


def _run_table() -> None:
    from mat_mul_b200 import _lib

    assert os.environ.get("CUDA_VISIBLE_DEVICES") == "", "the table runs only where no device is visible"
    L = _lib.lib()
    print(json.dumps({label: getattr(L, fn)(*args) for label, fn, args, _ in table()}))


def test_argument_rules_of_the_box_generators():
    res = subprocess.run([sys.executable, "-c", "from tests.test_box_ref import _run_table; _run_table()"], cwd=ROOT,
                         env={**os.environ, "CUDA_VISIBLE_DEVICES": ""}, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    got = json.loads(res.stdout.strip().splitlines()[-1])
    want = {label: w for label, _, _, w in table()}
    bad = {k: (got.get(k), w) for k, w in want.items() if got.get(k) != w}
    assert not bad, bad
