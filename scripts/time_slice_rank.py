"""tg_slice_rank at 9x9x9 and 25x25x25 on bench-like states, with CUDA events.

States: the targets of synthetic demos (coefficients -2..2 at 9x9x9 rank 23, -1..1 at 25x25x25 rank 100) and the
same games half played out; plus int8 slabs across the full range, where the rank needs more than one prime.
Prints the card and its power limit first; run on the GPU:  python scripts/time_slice_rank.py
"""
from __future__ import annotations

import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from mat_mul_b200 import env  # noqa: E402


def timed(fn, iters: int = 20, warmup: int = 3) -> float:
    """Seconds per call (CUDA events around `iters` back-to-back calls after `warmup` calls)."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / 1e3 / iters


def main() -> None:
    assert torch.cuda.is_available(), "time_slice_rank.py measures on the GPU"
    dev = torch.device("cuda:0")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print(f"card: {q[0] if q else torch.cuda.get_device_name(dev)}  (name, power limit, max SM clock)")
    for S, N, R, values, probs, shift in [(9, 1 << 20, 23, (-2, -1, 0, 1, 2), (0.05, 0.10, 0.70, 0.10, 0.05), 2),
                                          (25, 1 << 15, 100, (-1, 0, 1), (0.15, 0.7, 0.15), 1)]:
        tape, slab, _ = env.make_synthetic_demos(N, R, S, values, probs, shift, seed=3, device=dev)
        half, _, _ = env.replay(slab, tape[: R // 2].contiguous(), S, shift)
        g = torch.Generator(device=dev).manual_seed(S)
        full = torch.randint(-128, 128, slab.shape, dtype=torch.int8, device=dev, generator=g)
        full = env.pack_states(env.expand_states(full, S), S)  # zero padding
        for name, st in (("demo targets", slab), ("half played", half), ("int8 full range", full)):
            t = timed(lambda: env.slice_rank(st, S))
            r = env.slice_rank(st, S).float().mean().item()
            print(f"S={S:2d} {name:16s} {N} games: {t * 1e3:8.3f} ms  {N / t / 1e9:6.3f} G games/s  mean rank {r:.2f}")


if __name__ == "__main__":
    main()
