"""Synthetic demonstrations modulo 2: (a) tg_demo_gen_gf2 against (b) tg_demo_gen_philox + tg_pack_gf2, the route it
replaces, and (c) tg_demo_gen_philox alone, alternated in one run with CUDA events.  The device-to-device copy bandwidth
is measured in the same run.

Outputs are above the 126 MB L2: 2^22 / 2^20 / 2^18 / 2^16 demos at R = 7 / 23 / 49 / 100 for S = 4 / 9 / 16 / 25 (0.5
to 1.1 GB of tape and targets per call), each shape warmed up before its timed window, for the reference alphabet
{-1, 0, 1} and for V5 = {-2..2}.  Bytes per demo are the traffic the formats imply: (a) writes R TP + GB, (b) writes
R TP + GP, reads GP and writes GB, (c) writes R TP + GP.  Before timing, the tape and bits of (a) and (b) are compared at
{-1, 0, 1} (where they are the same demos).  Prints the card and its power limit first; run on the GPU:
    python scripts/time_gf2_demos.py > profiles/gf2_demos_time.txt
"""
from __future__ import annotations

import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from mat_mul_b200 import env  # noqa: E402

SHAPES = {4: (1 << 22, 7), 9: (1 << 20, 23), 16: (1 << 18, 49), 25: (1 << 16, 100)}
ALPHABETS = {"{-1,0,1}": ((-1, 0, 1), (0.15, 0.7, 0.15), 1), "V5": ((-2, -1, 0, 1, 2), (0.05, 0.10, 0.70, 0.10, 0.05), 2)}


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


def main() -> None:
    assert torch.cuda.is_available(), "time_gf2_demos.py measures on the GPU"
    dev = torch.device("cuda:0")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print(f"card: {q[0] if q else torch.cuda.get_device_name(dev)}  (name, power limit, max SM clock)")
    src = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
    dst = torch.empty_like(src)
    copy_bw = 2 * src.numel() / timed(lambda: dst.copy_(src), 10)
    print(f"device-to-device copy of 1 GiB: {copy_bw / 1e9:.0f} GB/s (read + write)")
    del src, dst
    print("(a) tg_demo_gen_gf2, (b) tg_demo_gen_philox + tg_pack_gf2, (c) tg_demo_gen_philox alone; best of 3 alternating rounds")
    print(f"{'path':30s} {'alphabet':9s} {'S':>3s} {'N':>8s} {'R':>4s} {'demos/s':>10s} {'B/demo':>7s} {'GB/s':>6s} {'of copy':>8s} "
          f"{'(b)/(a)':>8s}")
    for name, (values, probs, shift) in ALPHABETS.items():
        for S, (N, R) in SHAPES.items():
            lay, lb = env.layout(S), env.layout_gf2(S)
            tape = torch.empty((R, N, lay.token_pitch), dtype=torch.uint8, device=dev)
            slab = torch.empty((N, lay.game_pitch), dtype=torch.int8, device=dev)
            bits = torch.empty((N, lb.game_words), dtype=torch.int32, device=dev)
            kw = dict(seed=S, device=dev)
            if name == "{-1,0,1}":
                env.make_synthetic_demos(N, R, S, values, probs, shift, tape=tape, slab=slab, **kw)
                tape_a = tape.clone()
                env.make_synthetic_demos_gf2(N, R, S, values, probs, shift, tape=tape_a, bits=bits, **kw)
                assert torch.equal(tape_a, tape) and torch.equal(bits, env.pack_gf2(slab, S)), S
                del tape_a

            def run_a():
                env.make_synthetic_demos_gf2(N, R, S, values, probs, shift, tape=tape, bits=bits, **kw)

            def run_c():
                env.make_synthetic_demos(N, R, S, values, probs, shift, tape=tape, slab=slab, **kw)

            def run_b():
                run_c()
                env._call("tg_pack_gf2", (slab, bits), env._p(slab), env._p(bits), N, S)  # into the same bit slab as (a)

            best = {"a": 1e9, "b": 1e9, "c": 1e9}
            for _ in range(3):
                for k, f in (("a", run_a), ("b", run_b), ("c", run_c)):
                    best[k] = min(best[k], timed(f, 5))
            rec = R * lay.token_pitch
            nbytes = {"a": rec + lb.game_bytes, "b": rec + 2 * lay.game_pitch + lb.game_bytes, "c": rec + lay.game_pitch}
            for k, label in (("a", "(a) tg_demo_gen_gf2"), ("b", "(b) gen_philox + pack_gf2"), ("c", "(c) gen_philox alone")):
                t = best[k]
                ratio = f"{best['b'] / best['a']:8.2f}" if k == "a" else ""
                print(f"{label:30s} {name:9s} {S:3d} {N:8d} {R:4d} {N / t:10.4g} {nbytes[k]:7d} {N * nbytes[k] / t / 1e9:6.0f} "
                      f"{N * nbytes[k] / t / copy_bw:8.2f} {ratio}")
            del tape, slab, bits
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
