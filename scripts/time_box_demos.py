"""Demonstrations in the box of a rectangular product: tg_demo_gen_box and tg_demo_gen_box_gf2 beside the cubic
generators tg_demo_gen_philox and tg_demo_gen_gf2 at the same S, R and alphabet, alternated in one run with CUDA events.

Shapes and R (the best known ranks): <2,2,2>@4 R=7, <3,3,3>@9 R=23, <2,3,4>@16 R=20, <4,4,4>@16 R=49, <3,4,5>@25 R=47,
<5,5,5>@25 R=98, alphabet {-1, 0, 1}.  N is chosen so that tape and targets of one call take about 1 GB, above the
126 MB L2.  Each shape is warmed up before its timed window; best of 3 alternating rounds.  The split of tg_demo_gen_box
into its sampler (demo_box_sample_kernel) and its sum (the kernels tg_demo_accumulate picks) comes from torch.profiler
in a separate pass.  Prints the card and its power limit first; run on the GPU:
    python scripts/time_box_demos.py > profiles/box_demos_time.txt
"""
from __future__ import annotations

import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from mat_mul_b200 import env  # noqa: E402

CASES = [((2, 2, 2), 7), ((3, 3, 3), 23), ((2, 3, 4), 20), ((4, 4, 4), 49), ((3, 4, 5), 47), ((5, 5, 5), 98)]
VALUES, PROBS, SHIFT = (-1, 0, 1), (0.15, 0.7, 0.15), 1
BYTES = 1 << 30


def timed(fn, iters: int, warmup: int = 2) -> float:
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


def kernel_split(fn, iters: int = 3) -> tuple[float, float]:
    """(sampler, sum) device seconds per call of a tg_demo_gen_box call, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile

    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            fn()
        torch.cuda.synchronize()
    samp = summ = 0.0
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        t = e.cuda_time_total if t is None else t
        if "demo_box_sample_kernel" in e.key:
            samp += t
        elif "demo" in e.key:
            summ += t
    return samp / 1e6 / iters, summ / 1e6 / iters


def main() -> None:
    assert torch.cuda.is_available(), "time_box_demos.py measures on the GPU"
    dev = torch.device("cuda:0")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print(f"card: {q[0] if q else torch.cuda.get_device_name(dev)}  (name, power limit, max SM clock)")
    print(f"alphabet {VALUES} {PROBS}; best of 3 alternating rounds; sampler / sum split from torch.profiler (separate pass)")
    print(f"{'shape':9s} {'S':>3s} {'box':>12s} {'R':>4s} {'N':>8s} | {'box demos/s':>11s} {'sampler ms':>10s} {'sum ms':>7s} "
          f"{'philox demos/s':>14s} | {'box_gf2 demos/s':>15s} {'gf2 demos/s':>11s}")
    for (n, m, p), R in CASES:
        S, box = env.matmul_box(n, m, p)
        lay, lb = env.layout(S), env.layout_gf2(S)
        N = BYTES // (R * lay.token_pitch + lay.game_pitch)
        tape = torch.empty((R, N, lay.token_pitch), dtype=torch.uint8, device=dev)
        slab = torch.empty((N, lay.game_pitch), dtype=torch.int8, device=dev)
        bits = torch.empty((N, lb.game_words), dtype=torch.int32, device=dev)
        args = (VALUES, PROBS, SHIFT)
        runs = {
            "box": lambda: env.make_synthetic_demos_box(N, R, S, box, *args, seed=S, device=dev, tape=tape, slab=slab),
            "philox": lambda: env.make_synthetic_demos(N, R, S, *args, seed=S, device=dev, tape=tape, slab=slab),
            "box_gf2": lambda: env.make_synthetic_demos_box_gf2(N, R, S, box, *args, seed=S, device=dev, tape=tape, bits=bits),
            "gf2": lambda: env.make_synthetic_demos_gf2(N, R, S, *args, seed=S, device=dev, tape=tape, bits=bits),
        }
        best = {k: 1e9 for k in runs}
        for _ in range(3):
            for k, f in runs.items():
                best[k] = min(best[k], timed(f, 5))
        samp, summ = kernel_split(runs["box"])
        print(f"<{n},{m},{p}>  {S:3d} {str(box):>12s} {R:4d} {N:8d} | {N / best['box']:11.4g} {samp * 1e3:10.3f} {summ * 1e3:7.3f} "
              f"{N / best['philox']:14.4g} | {N / best['box_gf2']:15.4g} {N / best['gf2']:11.4g}")
        del tape, slab, bits
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
