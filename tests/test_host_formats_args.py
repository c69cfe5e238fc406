"""Argument rules of the host-buffer entry points (tg_*_host, int8, int16 and bit slabs) that hold without a device.

A null context, a negative batch or K, and a null host pointer are refused before the context is read; an empty batch
returns TG_OK before any pointer is looked at.  The table runs in a child process that sees no CUDA device, with a
context pointer that is never dereferenced: a check that is missing shows up as a crash or as TG_E_CUDA instead of the
expected code.
"""
import json
import os
import subprocess
import sys

from mat_mul_b200 import _lib
from tests.test_cabi_args import E_ARG, OK, ROOT, ptr

STEP = ("ctx", "in", "tape", "out", "flags", "nnz", "B", "shift")
ROLLOUT = ("ctx", "in", "tape", "K", "out", "flags", "nnz", "steps", "B", "shift")
DEMO = ("ctx", "seed", "first", "B", "R", "shift", "values", "probs", "n_values", "max_tries", "tape", "out", "flags")
VALID = dict(B=4, K=3, R=5, shift=2, seed=1, first=0, n_values=3, max_tries=8)
SUFFIXES = ("", "_i16", "_gf2")


def table():
    """(label, entry point, arguments, expected code); each row breaks one argument and keeps the others valid."""
    n = None
    rows = []

    def add(fn, names, label, expect, **kw):
        a = {**VALID, **kw}
        rows.append((f"{fn} {label}", fn, tuple(a[k] if k in a else ptr() for k in names), expect))

    shapes = [(f"tg_step_host{s}", STEP) for s in SUFFIXES] + [(f"tg_rollout_host{s}", ROLLOUT) for s in SUFFIXES]
    shapes += [(f"tg_demo_gen_host{s}", DEMO) for s in ("", "_gf2")]
    for fn, names in shapes:
        ptrs = [k for k in names if k not in VALID and k != "ctx"]
        add(fn, names, "null context", E_ARG, ctx=n)
        add(fn, names, "null context, empty batch", E_ARG, ctx=n, B=0)
        add(fn, names, "B -1", E_ARG, B=-1)
        add(fn, names, "empty batch, null pointers", OK, B=0, **{k: n for k in ptrs})
        for k in ptrs:
            if names is ROLLOUT and k == "tape":
                add(fn, names, "null tape", E_ARG, tape=n)  # K = 3 needs one; K = 0 would go on to the device
            elif names is not DEMO or k not in ("values", "probs"):  # the demo generator checks those itself
                add(fn, names, f"null {k}", E_ARG, **{k: n})
        if names is ROLLOUT:
            add(fn, names, "K -1", E_ARG, K=-1)
            add(fn, names, "empty batch, K -1", E_ARG, B=0, K=-1)
        if names is DEMO:
            add(fn, names, "R 0", E_ARG, R=0)
            add(fn, names, "empty batch, R 0", E_ARG, B=0, R=0)
    return rows


def _run_table() -> None:
    """Child process: every row's return code, as JSON on stdout."""
    assert os.environ.get("CUDA_VISIBLE_DEVICES") == "", "the table runs only where no device is visible"
    L = _lib.lib()
    print(json.dumps({label: getattr(L, fn)(*args) for label, fn, args, _ in table()}))


def test_host_entry_points_are_declared_and_bound():
    names = {r[1] for r in table()}
    assert len(names) == 8 and names <= set(_lib.exported_symbols()) and names <= set(_lib._SIGNATURES)


def test_argument_rules_of_the_host_entry_points():
    rows = table()
    assert len({r[0] for r in rows}) == len(rows)
    res = subprocess.run([sys.executable, "-c", "from tests.test_host_formats_args import _run_table; _run_table()"], cwd=ROOT,
                         env={**os.environ, "CUDA_VISIBLE_DEVICES": ""}, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr
    got = json.loads(res.stdout.strip().splitlines()[-1])
    wrong = [f"{label}: {got[label]}, want {want}" for label, _, _, want in rows if got[label] != want]
    assert not wrong, f"{len(wrong)} of {len(rows)} calls:\n" + "\n".join(wrong)
