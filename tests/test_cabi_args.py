"""Argument rules of the C entry points at every size: the game path for the int8, int16 and bit-slab twins, and the
demo generators, accumulations, sample batchers, tape transpose and changes of basis over Z and GF(2).

Every call in the table must be refused by the library's own checks (TG_E_ARG) or be an empty batch (TG_OK); none may
launch.  The table runs in a child process that sees no CUDA device, so a check that is missing shows up as TG_E_CUDA
(-2, the call got past its checks and tried to reach the device) instead of a launch on a pointer that is not one.
Host arrays (the demo alphabets) are real, so a call that gets past its checks can read them.
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
BASIS_SIZES = (4, 9, 16)  # the change of basis over Z
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


# the demo alphabet (host arrays): int8 values with float64 probabilities, or float32 for tg_demo_from_ustream
VALUES = (C.c_int8 * 3)(-1, 0, 1)
PROBS = (C.c_double * 3)(0.15, 0.7, 0.15)
PROBS_F32 = (C.c_float * 3)(0.15, 0.7, 0.15)


# argument names of each shape, in C order (stream last); shared by the three formats' twins
STEP = ("in", "tape", "out", "flags", "nnz", "B", "S", "shift", "stream")
EXPAND = ("in", "tape", "k", "out", "flags", "nnz", "keys", "B", "S", "shift", "stream")
ROLLOUT = ("in", "tape", "stride", "K", "out", "flags", "nnz", "steps", "B", "S", "shift", "stream")
REPLAY = tuple(a for a in ROLLOUT if a != "steps")
PAIR = ("src", "dst", "B", "S", "stream")
PACK_F32 = ("src", "ld", "dst", "B", "S", "flag", "stream")
EXPAND_F32 = ("src", "dst", "ld", "B", "S", "stream")
PACK_ACTIONS = ("src", "dst", "B", "S", "flag", "stream")
# B is the batch that may be empty (N of the demo and basis calls, nb of the sample batchers)
DEMO_GEN = ("seed", "first", "B", "R", "S", "shift", "values", "probs", "n_values", "max_tries", "tape", "stride", "out", "flags",
            "stream")
ACCUMULATE = ("tape", "stride", "B", "R", "S", "shift", "out", "flags", "stream")
USTREAM = ("u", "n_u", "values", "probs_f32", "n_values", "R", "S", "shift", "B", "tape", "stride", "out", "flags", "result", "ws",
           "ws_bytes", "stream")
SAMPLE = ("tape", "stride", "targets", "N", "R", "S", "dim_t", "replay_shift", "idx", "B", "states", "scalars", "actions", "rewards",
          "stream")
SAMPLE_DM = ("tape", "targets", "t16", "bound", "N", "R", "S", "dim_t", "replay_shift", "idx", "B", "states", "scalars", "actions",
             "rewards", "stream")
SAMPLE_GF2 = ("tape", "targets", "N", "R", "S", "dim_t", "replay_shift", "idx", "B", "states", "scalars", "actions", "rewards", "stream")
SAMPLE_PTRS = ("tape", "targets", "idx", "states", "scalars", "actions", "rewards")
TRANSPOSE = ("tape", "stride", "out", "B", "R", "S", "stream")
BASIS = ("in", "mats", "per_game", "out", "flags", "B", "S", "stream")
BASIS_GF2 = tuple(a for a in BASIS if a != "flags")
FACTORS = ("tape", "stride", "shift_in", "mats", "per_game", "out", "out_stride", "shift_out", "flags", "B", "R", "S", "stream")
FACTORS_GF2 = tuple(a for a in FACTORS if a != "flags")
SAMPLE_MATS = ("seed", "first", "B", "S", "p", "mats", "stream")
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
    valid = dict(B=4, S=S, shift=2, k=3, K=2, stride=32, ld=S ** 3, keys=n, flag=n, stream=n, seed=1, first=0, R=2, n_values=3,
                 max_tries=8, values=C.c_void_p(C.addressof(VALUES)), probs=C.c_void_p(C.addressof(PROBS)),
                 probs_f32=C.c_void_p(C.addressof(PROBS_F32)), out=ptr(4096), n_u=3 * S * 10, ws_bytes=1 << 30, N=8, dim_t=2,
                 replay_shift=2, t16=0, bound=127, per_game=1, out_stride=32, shift_in=2, shift_out=2, p=0.3)
    out = []

    def add(fn, names, label, expect, sizes=SIZES, **kw):
        a = {**valid, **kw}
        args = tuple(a[k] if k in a else ptr() for k in names)
        out.append((f"{fn} S={S} {label}", fn, args, expect if S in sizes else E_ARG))  # every call fails at a bad S

    def common(fn, names, pointers, aligned, sizes=SIZES):
        if S not in sizes:
            add(fn, names, "otherwise valid", E_ARG, sizes)  # at a supported S this call would launch
        add(fn, names, "empty batch", OK, sizes, B=0, **{k: n for k in pointers})
        add(fn, names, "B -1", E_ARG, sizes, B=-1)
        add(fn, names, "all null", E_ARG, sizes, **{k: n for k in pointers})
        for k in pointers:
            add(fn, names, f"{k} null", E_ARG, sizes, **{k: n})
        for k, align in aligned.items():
            for o in (1, 2, 4, 8):
                if o % align:
                    add(fn, names, f"{k} at +{o}", E_ARG, sizes, **{k: ptr(o)})

    def bad(fn, names, sizes=SIZES, **edges):
        """each scalar just outside its range, alone and with an empty batch (a bad scalar is refused first)"""
        for k, vals in edges.items():
            for v in vals:
                add(fn, names, f"{k} {v}", E_ARG, sizes, **{k: v})
                add(fn, names, f"empty batch, {k} {v}", E_ARG, sizes, B=0, **{k: v})

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

    def strides(fn, names, key="stride", sizes=SIZES):
        for st in (4, 8, 40):
            add(fn, names, f"{key} {st}", E_ARG, sizes, **{key: st})

    for fn in ("tg_demo_gen_philox", "tg_demo_gen_gf2"):
        common(fn, DEMO_GEN, ("values", "probs", "tape", "out"), {"tape": 16, "out": 16})
        bad(fn, DEMO_GEN, R=(0, 65536), shift=(0, 5), n_values=(0, 9), max_tries=(0, 65536))
        strides(fn, DEMO_GEN)
    for fn, shifts, sizes in (("tg_demo_accumulate", (0, 5), SIZES), ("tg_demo_accumulate_i16", (-1, 128), SIZES),
                              ("tg_demo_accumulate_tc", (0, 5), (16,))):
        common(fn, ACCUMULATE, ("tape", "out"), {"tape": 16, "out": 16}, sizes)
        bad(fn, ACCUMULATE, sizes, R=(0, 65) if sizes == (16,) else (0,), shift=shifts)
        strides(fn, ACCUMULATE, sizes=sizes)
    fn = "tg_demo_from_ustream"
    common(fn, USTREAM, ("u", "values", "probs_f32", "tape", "out", "result", "ws"), {"tape": 16, "out": 16, "ws": 16})
    bad(fn, USTREAM, R=(0,), shift=(0, 5), n_values=(0, 9), n_u=(-1, 3 * S << 31))
    strides(fn, USTREAM)
    add(fn, USTREAM, "workspace too small", E_ARG, ws_bytes=64)

    # tg_demo_sample: the step-major records may start anywhere and any replay_shift goes (int32 lanes outside [0, 8])
    common("tg_demo_sample", SAMPLE, SAMPLE_PTRS, {"targets": 16})
    bad("tg_demo_sample", SAMPLE, N=(-1,), R=(0,), dim_t=(0,))
    for fn, names in (("tg_demo_sample_dm", SAMPLE_DM), ("tg_demo_sample_gf2", SAMPLE_GF2)):
        common(fn, names, SAMPLE_PTRS, {"tape": 16, "targets": 16})
        bad(fn, names, N=(-1,), R=(0,), dim_t=(0,), **({"bound": (-1,)} if "bound" in names else {}))
        for sh in (-1, 9):  # tested after the pointers: an empty batch with this shift is accepted
            add(fn, names, f"replay_shift {sh}", E_ARG, replay_shift=sh)
            add(fn, names, f"empty batch, replay_shift {sh}", OK, B=0, replay_shift=sh)
    common("tg_tape_to_demo_major", TRANSPOSE, ("tape", "out"), {"tape": 16, "out": 16})
    bad("tg_tape_to_demo_major", TRANSPOSE, R=(0,))
    strides("tg_tape_to_demo_major", TRANSPOSE)

    # the change of basis: int8 matrices at any address over Z, uint32 rows over GF(2)
    for fn in ("tg_change_of_basis", "tg_change_of_basis_i16"):
        common(fn, BASIS, ("in", "mats", "out"), {"in": 16, "out": 16}, BASIS_SIZES)
        add(fn, BASIS, "in place", E_ARG, BASIS_SIZES, out=ptr())
    common("tg_change_of_basis_gf2", BASIS_GF2, ("in", "mats", "out"), {"in": 16, "out": 16, "mats": 4})
    fn = "tg_change_of_basis_factors"
    common(fn, FACTORS, ("tape", "mats", "out", "flags"), {"tape": 16}, BASIS_SIZES)
    bad(fn, FACTORS, BASIS_SIZES, R=(0,), shift_in=(-1,), shift_out=(0, 128))
    strides(fn, FACTORS, sizes=BASIS_SIZES)
    fn = "tg_change_of_basis_factors_gf2"
    common(fn, FACTORS_GF2, ("tape", "mats", "out"), {"tape": 16, "out": 16, "mats": 4})
    bad(fn, FACTORS_GF2, R=(0,), shift_in=(0, 5), shift_out=(0, 5))
    strides(fn, FACTORS_GF2)
    strides(fn, FACTORS_GF2, "out_stride")
    for fn, align, sizes in (("tg_sample_unimodular", 1, BASIS_SIZES), ("tg_sample_invertible_gf2", 4, SIZES)):
        common(fn, SAMPLE_MATS, ("mats",), {"mats": align}, sizes)
        bad(fn, SAMPLE_MATS, sizes, p=(-0.01, 1.01, float("nan")))
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
