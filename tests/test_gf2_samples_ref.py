"""The mod-2 training samples without a GPU: tests/gf2_samples_ref.py pinned to the C oracle's integer sample taken mod 2
(tests/oracle_any_s.py at 25), and the argument rules of tg_demo_sample_gf2 and tg_expand_f32_gf2."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from mat_mul_b200 import _lib
from oracle import tg_oracle as orc
from tests import gf2_samples_ref as ref
from tests import oracle_any_s
from tests.test_cabi_args import BAD_SIZES, E_ARG, OK, ROOT, ptr

SIZES = (4, 9, 16, 25)
SHIFTS = (0, 1, 2, 8)
R = 7


@pytest.mark.parametrize("S", SIZES)
@pytest.mark.parametrize("replay_shift", SHIFTS)
def test_sample_is_the_oracle_sample_mod_2(S, replay_shift):
    rng = np.random.default_rng(S * 10 + replay_shift)
    getitem = oracle_any_s.demo_getitem if S == 25 else orc.demo_getitem
    tok = rng.integers(0, 9, size=(R, 3 * S))
    target = rng.integers(-9, 10, size=(S, S, S))
    for dim_t in (1, 2, 4, R + 2):
        for a in (0, R - 1, int(rng.integers(1, R - 1))):
            want = np.asarray(getitem(tok, target, dim_t, a, replay_shift=replay_shift)[0], dtype=np.int64) & 1
            assert np.array_equal(ref.demo_getitem(tok, target, dim_t, a, replay_shift), want), (dim_t, a)


@pytest.mark.parametrize("S", SIZES)
def test_batch_is_the_sample_of_every_index(S):
    rng = np.random.default_rng(S)
    N = 3
    tok = rng.integers(0, 256, size=(N, R, 3 * S))
    targets = rng.integers(-5, 6, size=(N, S, S, S))
    idx = np.array([0, N * R - 1, -1, N * R, 9, R - 1, R, 1 << 40])
    for dim_t in (1, 3, R + 2):
        st, sc, ac, rw, valid = ref.samples(tok, targets, idx, dim_t, 1)
        assert valid.tolist() == [True, True, False, False, True, True, True, False]
        assert not st[~valid].any() and st.max() <= 1
        for b in np.flatnonzero(valid):
            d, a = divmod(int(idx[b]), R)
            assert np.array_equal(st[b], ref.demo_getitem(tok[d], targets[d], dim_t, a, 1)), (dim_t, b)
            assert sc[b, 0] == R - a and rw[b, 0] == -(a + 1) and np.array_equal(ac[b], tok[d, a])


# ---------------------------------------------------------------- argument rules
SAMPLE = ("tape", "targets", "N", "R", "S", "dim_t", "replay_shift", "idx", "nb", "states", "scalars", "actions", "rewards", "stream")
EXPAND = ("src", "dst", "ld", "B", "S", "stream")
SAMPLE_PTRS = ("tape", "targets", "idx", "states", "scalars", "actions", "rewards")


def _rows(S: int):
    """(label, entry point, arguments, expected code); each row breaks one argument and keeps the others valid."""
    n = None
    valid = dict(N=4, R=3, S=S, dim_t=2, replay_shift=1, nb=5, ld=S ** 3, B=4, stream=n)
    out = []

    def add(fn, names, label, expect, **kw):
        a = {**valid, **kw}
        out.append((f"{fn} S={S} {label}", fn, tuple(a[k] if k in a else ptr() for k in names), expect if S in SIZES else E_ARG))

    fn = "tg_demo_sample_gf2"
    if S not in SIZES:
        add(fn, SAMPLE, "otherwise valid", E_ARG)
    add(fn, SAMPLE, "empty batch", OK, nb=0, **{k: n for k in SAMPLE_PTRS})
    add(fn, SAMPLE, "empty batch, replay_shift 9", OK, nb=0, replay_shift=9)  # replay_shift is checked after the pointers
    for k, bad in (("N", -1), ("R", 0), ("R", -1), ("dim_t", 0), ("dim_t", -1), ("nb", -1)):
        add(fn, SAMPLE, f"{k} {bad}", E_ARG, **{k: bad})
        add(fn, SAMPLE, f"{k} {bad}, empty batch", E_ARG, **{k: bad}, **({} if k == "nb" else {"nb": 0}))
    for sh in (-1, 9, 100):
        add(fn, SAMPLE, f"replay_shift {sh}", E_ARG, replay_shift=sh)
    add(fn, SAMPLE, "all null", E_ARG, **{k: n for k in SAMPLE_PTRS})
    for k in SAMPLE_PTRS:
        add(fn, SAMPLE, f"{k} null", E_ARG, **{k: n})
    for k in ("tape", "targets"):
        for o in (1, 2, 4, 8):
            add(fn, SAMPLE, f"{k} at +{o}", E_ARG, **{k: ptr(o)})
    add(fn, SAMPLE, "null idx, replay_shift 9", E_ARG, idx=n, replay_shift=9)

    fn = "tg_expand_f32_gf2"
    if S not in SIZES:
        add(fn, EXPAND, "otherwise valid", E_ARG)
    add(fn, EXPAND, "empty batch", OK, B=0, src=n, dst=n)
    add(fn, EXPAND, "B -1", E_ARG, B=-1)
    add(fn, EXPAND, "all null", E_ARG, src=n, dst=n)
    for k in ("src", "dst"):
        add(fn, EXPAND, f"{k} null", E_ARG, **{k: n})
    for o in (1, 2, 4, 8):
        add(fn, EXPAND, f"bits at +{o}", E_ARG, src=ptr(o))
    for o in (1, 2, 3):
        add(fn, EXPAND, f"dst at +{o}", E_ARG, dst=ptr(o))
    return out


def table():
    return [r for S in SIZES + BAD_SIZES for r in _rows(S)]


def _run_table() -> None:
    """Child process: every row's return code, as JSON on stdout."""
    assert os.environ.get("CUDA_VISIBLE_DEVICES") == "", "the table runs only where no device is visible"
    L = _lib.lib()
    print(json.dumps({label: getattr(L, fn)(*args) for label, fn, args, _ in table()}))


def test_argument_rules_of_the_mod_2_samples():
    rows = table()
    assert len({r[0] for r in rows}) == len(rows)
    res = subprocess.run([sys.executable, "-c", "from tests.test_gf2_samples_ref import _run_table; _run_table()"], cwd=ROOT,
                         env={**os.environ, "CUDA_VISIBLE_DEVICES": ""}, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr
    got = json.loads(res.stdout.strip().splitlines()[-1])
    wrong = [f"{label}: {got[label]}, want {want}" for label, _, _, want in rows if got[label] != want]
    assert not wrong, f"{len(wrong)} of {len(rows)} calls:\n" + "\n".join(wrong)
