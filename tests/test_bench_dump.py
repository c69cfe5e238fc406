"""bench.py --dump-outputs: the files hold what the last timed step returned (checked against the oracle), --steps sets
how many steps ran, and arrays over the budget keep one fixed, seeded sample of games."""
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from oracle import tg_oracle as orc
from tests.helpers import dense_to_slab, tokens_to_tape3

ROOT = Path(__file__).resolve().parents[1]
V5, P5 = (-2, -1, 0, 1, 2), (0.05, 0.10, 0.70, 0.10, 0.05)  # bench.py's VALUES5 / PROBS5
SHIFT, B = 2, 4096


def _bench(out: Path, *args: str) -> dict:
    cmd = [sys.executable, str(ROOT / "bench.py"), "--games", str(B), "--no-e2e", "--no-cpu", "--no-extras", *args,
           "--dump-outputs", str(out)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    got = {p.stem: np.load(p) for p in out.glob("*.npy")}
    assert all(a.dtype == np.float32 for a in got.values())
    assert sum(p.stat().st_size for p in out.glob("*.npy")) <= 64_000_000
    return got


def _range_flag(T: np.ndarray) -> np.ndarray:
    """TG_FLAG_RANGE (4) for every game with an entry outside [-64, 63]."""
    return np.where((np.abs(T.reshape(T.shape[0], -1) + 0.5) > 64).any(1), 4, 0)


def _replayed(S: int, R: int, n_steps: int):
    """The bench's games (seed 0x5EED) after n_steps of their demos replayed in reverse, with the last step's full flags
    (the oracle's TERMINAL / NULL bits and the range bit) and nnz."""
    tok, cur, ex = orc.demos_philox(0x5EED, 0, B, V5, P5, R, S, SHIFT)
    assert ex == 0
    for i in range(n_steps):
        cur, flags, nnz = orc.step_batch(cur, tok[:, R - 1 - i], SHIFT)
    return dense_to_slab(cur), flags | _range_flag(cur), nnz


@pytest.mark.gpu
@pytest.mark.parametrize("steps", [1, 4, 18])  # after 5 + 18 = R steps every game is terminal (flags 1)
def test_step_dump_is_the_last_timed_step(tmp_path, steps):
    np.save(tmp_path / "tape.npy", np.zeros(3, np.float32))  # left by an earlier --metric demos dump into the same DIR
    got = _bench(tmp_path, "--steps", str(steps), "--warmup", "5")
    assert set(got) == {"slab", "flags", "nnz"}
    slab, flags, nnz = _replayed(9, 23, 5 + steps)
    assert np.array_equal(got["slab"], slab) and np.array_equal(got["nnz"], nnz) and np.array_equal(got["flags"], flags)


@pytest.mark.gpu
def test_dump_over_budget_keeps_a_seeded_sample(tmp_path):
    got = _bench(tmp_path, "--size", "16", "--steps", "2", "--warmup", "3")
    n = 60_000_000 // ((4096 + 2) * 4)  # bench.py's DUMP_BYTES over the float32 bytes of one 16x16x16 game's outputs
    idx = np.sort(np.random.default_rng(0).choice(B, n, replace=False))
    slab, flags, nnz = _replayed(16, 49, 5)
    assert np.array_equal(got["slab"], slab[idx]) and np.array_equal(got["nnz"], nnz[idx])
    assert np.array_equal(got["flags"], flags[idx])


@pytest.mark.gpu
def test_demo_dump_is_the_last_timed_launch(tmp_path):
    got = _bench(tmp_path, "--metric", "demos", "--steps", "2", "--warmup", "0")
    assert set(got) == {"tape", "slab", "flags"}
    tok, tgt, ex = orc.demos_philox(0xD0 + 1, 0, B, V5, P5, 23, 9, SHIFT)  # launch i draws seed 0xD0 + i
    assert ex == 0  # no term needed the forced unit triple, so TG_FLAG_EXHAUSTED (8) is never due
    assert np.array_equal(got["tape"], tokens_to_tape3(tok)) and np.array_equal(got["slab"], dense_to_slab(tgt))
    assert np.array_equal(got["flags"], _range_flag(tgt))


@pytest.mark.parametrize("args", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bench_rejects_bad_arguments(args):
    res = subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert res.returncode == 2 and "error" in res.stderr
