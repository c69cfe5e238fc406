"""Argument rules of the game path's C entry points, for the int8, int16 and bit-slab twins at every size.

Every call in the table must be refused by the library's own checks (TG_E_ARG) or be an empty batch (TG_OK); none may
launch.  The table runs in a child process that sees no CUDA device, so a check that is missing shows up as TG_E_CUDA
(-2, the call got past its checks and tried to reach the device) instead of a launch on a pointer that is not one.
"""
import ctypes as C
import json
import os
import subprocess
import sys
from pathlib import Path

from mat_mul_b200 import _lib

ROOT = Path(__file__).resolve().parents[1]
SIZES = (4, 9, 16, 25)
BAD_SIZES = (-4, 0, 1, 3, 5, 7, 8, 36)
OK, E_ARG = 0, -1

BASE = 1 << 20  # never dereferenced

# tg_expand_children*: threads per CTA of the word-column kernel (int8 at 4 uses a row kernel without shared memory)
EXPAND_NT = {"": {9: 128, 16: 128, 25: 160}, "_i16": {4: 128, 9: 256, 16: 256, 25: 320}}
EXPAND_SMEM_CAP = 200 * 1024  # bytes of shared memory the records and child stages of a CTA may take


def expand_limits(sfx: str, S: int):
    """(k whose TG * k * TP bytes of records is a multiple of 2^32, the first k whose records exceed shared memory)"""
    rp = (S * S + 3) & ~3
    gp, tp = (S * rp + 15) & ~15, (3 * S + 15) & ~15
    eb = 2 if sfx else 1
    nt = EXPAND_NT[sfx][S]
    tg = nt // (rp * eb // 4)
    smem0 = 3 * tg * gp * eb + ((3 * tg * 4 + 7) & ~7) + tg * 8 + 16 + nt * 8
    wrap = next(1 << e for e in range(1, 31) if (tg * tp << e) % (1 << 32) == 0)
    return wrap, (EXPAND_SMEM_CAP - smem0) // (tg * tp) + 1


def ptr(offset: int = 0) -> C.c_void_p:
    return C.c_void_p(BASE + offset)


# argument names of each shape, in C order (stream last); shared by the three formats' twins
STEP = ("in", "tape", "out", "flags", "nnz", "B", "S", "shift", "stream")
EXPAND = ("in", "tape", "k", "out", "flags", "nnz", "keys", "B", "S", "shift", "stream")
ROLLOUT = ("in", "tape", "stride", "K", "out", "flags", "nnz", "steps", "B", "S", "shift", "stream")
REPLAY = tuple(a for a in ROLLOUT if a != "steps")
PAIR = ("src", "dst", "B", "S", "stream")
PACK_F32 = ("src", "ld", "dst", "B", "S", "flag", "stream")
EXPAND_F32 = ("src", "dst", "ld", "B", "S", "stream")
PACK_ACTIONS = ("src", "dst", "B", "S", "flag", "stream")
# one source and one destination buffer per game: (entry points, argument names, source and destination alignment)
PAIRS = [(("tg_state_key", "tg_state_key_i16", "tg_state_key_gf2", "tg_slice_rank", "tg_slice_rank_i16", "tg_slice_rank_gf2"),
          PAIR, 16, 1),
         (("tg_pack_gf2", "tg_pack_gf2_i16", "tg_unpack_gf2"), PAIR, 16, 16),
         (("tg_pack_f32", "tg_pack_f32_i16"), PACK_F32, 4, 16),
         (("tg_expand_f32", "tg_expand_f32_i16"), EXPAND_F32, 16, 4),
         (("tg_pack_actions_i64",), PACK_ACTIONS, 8, 16),
         (("tg_unpack_actions_i64",), PAIR, 16, 8)]


def _rows(S: int):
    """(label, entry point, arguments, expected code) of every shape at one S.  A row names the argument it breaks;
    every other argument is valid, so only that one can make the call fail."""
    n = None
    valid = dict(B=4, S=S, shift=2, k=3, K=2, stride=32, ld=S ** 3, keys=n, flag=n, stream=n)
    out = []

    def add(fn, names, label, expect, **kw):
        a = {**valid, **kw}
        args = tuple(a[k] if k in a else ptr() for k in names)
        out.append((f"{fn} S={S} {label}", fn, args, expect if S in SIZES else E_ARG))  # every call fails at a bad S

    def common(fn, names, pointers, aligned):
        if S not in SIZES:
            add(fn, names, "otherwise valid", E_ARG)  # at a supported S this call would launch
        add(fn, names, "empty batch", OK, B=0, **{k: n for k in pointers})
        add(fn, names, "B -1", E_ARG, B=-1)
        add(fn, names, "all null", E_ARG, **{k: n for k in pointers})
        for k in pointers:
            add(fn, names, f"{k} null", E_ARG, **{k: n})
        for k, align in aligned.items():
            for o in (1, 2, 4, 8):
                if o % align:
                    add(fn, names, f"{k} at +{o}", E_ARG, **{k: ptr(o)})

    slabs16 = {"in": 16, "tape": 16, "out": 16}
    for sfx in ("", "_i16", "_gf2"):
        fn = "tg_step" + sfx
        common(fn, STEP, ("in", "tape", "out", "flags", "nnz"), slabs16)
        for sh in (0, 5, 9):
            add(fn, STEP, f"shift {sh}", E_ARG, shift=sh)
        add(fn, STEP, "empty batch, shift 0", E_ARG, B=0, shift=0)

        fn = "tg_expand_children" + sfx
        common(fn, EXPAND, ("in", "tape", "out", "flags", "nnz"), slabs16)
        for sh in (0, 5, 9):
            add(fn, EXPAND, f"shift {sh}", E_ARG, shift=sh)
        for k in (0, -1):
            add(fn, EXPAND, f"k {k}", E_ARG, k=k)
        add(fn, EXPAND, "empty batch, k 0", E_ARG, B=0, k=0)
        add(fn, EXPAND, "all null but keys", E_ARG, **{k: n for k in ("in", "tape", "out", "flags", "nnz")}, keys=ptr())
        if S in EXPAND_NT.get(sfx, {}):  # the records of a CTA must fit shared memory, also where their size wraps int
            wrap, over = expand_limits(sfx, S)
            for k in (wrap, over):
                for keys in (n, ptr()):
                    add(fn, EXPAND, f"k {k}{' with keys' if keys else ''}", E_ARG, k=k, keys=keys)

        for fn, names in (("tg_rollout" + sfx, ROLLOUT), ("tg_replay" + sfx, REPLAY)):
            common(fn, names, tuple(k for k in ("in", "out", "flags", "nnz", "steps") if k in names), slabs16)
            for sh in (0, 5, 9):
                add(fn, names, f"shift {sh}", E_ARG, shift=sh)
            add(fn, names, "K -1", E_ARG, K=-1)
            add(fn, names, "empty batch, K -1", E_ARG, B=0, K=-1)
            add(fn, names, "tape null with K 2", E_ARG, tape=n)
            for st in (4, 8, 40):
                add(fn, names, f"step stride {st}", E_ARG, stride=st)

    for fns, names, a_src, a_dst in PAIRS:
        for fn in fns:
            common(fn, names, ("src", "dst"), {"src": a_src, "dst": a_dst})
    return out


def table():
    return [r for S in SIZES + BAD_SIZES for r in _rows(S)]


def _run_table() -> None:
    """Child process: every row's return code, as JSON on stdout."""
    assert os.environ.get("CUDA_VISIBLE_DEVICES") == "", "the table runs only where no device is visible"
    L = _lib.lib()
    print(json.dumps({label: getattr(L, fn)(*args) for label, fn, args, _ in table()}))


def test_argument_rules_of_every_format_and_size():
    rows = table()
    assert len({r[0] for r in rows}) == len(rows)
    res = subprocess.run([sys.executable, "-c", "from tests.test_cabi_args import _run_table; _run_table()"], cwd=ROOT,
                         env={**os.environ, "CUDA_VISIBLE_DEVICES": ""}, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr
    got = json.loads(res.stdout.strip().splitlines()[-1])
    wrong = [f"{label}: {got[label]}, want {want}" for label, _, _, want in rows if got[label] != want]
    assert not wrong, f"{len(wrong)} of {len(rows)} calls:\n" + "\n".join(wrong)
