"""Rates of the 25x25x25 kernels (5x5 matrix multiplication) with CUDA events, against a device-to-device copy
measured in the same run.

Working sets are larger than the 126 MB L2 (2^16 games = 1.03 GB of slab), every shape is warmed up before its timed
window, and the bytes are the algorithmic traffic computed from the shapes (what the kernel must read and write at
least).  Prints the card and its power limit first; run on the GPU:  python scripts/time_s25.py > profiles/<name>.txt
"""
from __future__ import annotations

import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from mat_mul_b200 import env  # noqa: E402

S = 25
V3, P3 = (-1, 0, 1), (0.15, 0.7, 0.15)


def timed(fn, iters: int = 10, warmup: int = 2) -> float:
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
    assert torch.cuda.is_available(), "time_s25.py measures on the GPU"
    dev = torch.device("cuda:0")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print(f"card: {q[0] if q else torch.cuda.get_device_name(dev)}  (name, power limit, max SM clock)")
    lay = env.layout(S)
    GP, TP = lay.game_pitch, lay.token_pitch
    rows = []

    src = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
    dst = torch.empty_like(src)
    t = timed(lambda: dst.copy_(src))
    copy_bw = 2 * src.numel() / t
    print(f"device-to-device copy of 1 GiB: {copy_bw / 1e9:.0f} GB/s (read + write)")
    del src, dst

    def report(name, t, n, unit, nbytes, bound):
        rows.append((name, n / t, unit, nbytes / t, nbytes / t / copy_bw, bound))

    # demos: N = 2^16, R = 100 (reference-style distribution); the store the other kernels read
    N, R, shift = 1 << 16, 100, 1
    tape, slab, _ = env.make_synthetic_demos(N, R, S, V3, P3, shift, seed=1, device=dev)
    t = timed(lambda: env.make_synthetic_demos(N, R, S, V3, P3, shift, seed=1, device=dev, tape=tape, slab=slab), iters=3, warmup=1)
    report("tg_demo_gen_philox (v1, R=100)", t, N, "demos/s", R * N * TP + N * GP, "sampler (Philox + rejection) then column sum")
    t = timed(lambda: env.accumulate_demos(tape, S, shift, slab=slab), iters=3, warmup=1)
    report("tg_demo_accumulate (R=100)", t, N, "demos/s", R * N * TP + N * GP, "IMADs: 25 x 4 per thread and term")
    slab16, _ = env.accumulate_demos16(tape, S, shift)
    t = timed(lambda: env.accumulate_demos16(tape, S, shift, slab16=slab16), iters=3, warmup=1)
    report("tg_demo_accumulate_i16 (R=100)", t, N, "demos/s", R * N * TP + 2 * N * GP, "IMADs: 25 x 4 per thread and term")

    # K1: 2^16 games in, 2^16 games out
    B = 1 << 16
    tape1 = tape[0].contiguous()
    out = torch.empty_like(slab)
    t = timed(lambda: env.step_batch(slab, tape1, S, shift, out=out), iters=20)
    report("tg_step (K1)", t, B, "game-steps/s", B * (2 * GP + TP + 5), "HBM")
    # K2: 32 steps per game
    K = 32
    rev = tape[:K].flip(0).contiguous()
    t = timed(lambda: env.rollout(slab, rev, S, shift, out=out), iters=5)
    report(f"tg_rollout (K2, K={K})", t, B * K, "game-steps/s", 2 * B * GP + K * B * TP + 9 * B, "IMADs: 25 per thread and step")
    # K8: 2^13 parents x 8 children (1.03 GB of children)
    P, k = 1 << 13, 8
    tape_bk = tape[:k, :P].permute(1, 0, 2).contiguous()
    parents = slab[:P].contiguous()
    env.expand_children(parents, tape_bk, S, shift)
    t = timed(lambda: env.expand_children(parents, tape_bk, S, shift), iters=5)
    report(f"tg_expand_children (K8, k={k})", t, P * k, "children/s", P * GP + P * k * (GP + TP + 13), "HBM (one bulk store per child)")
    t = timed(lambda: env.state_keys(slab, S), iters=10)
    report("tg_state_key (K7)", t, B, "games/s", B * (GP + 8), "HBM")
    Br = 1 << 14
    sr = slab[:Br].contiguous()
    t = timed(lambda: env.slice_rank(sr, S), iters=5)
    report("tg_slice_rank (K6)", t, Br, "games/s", Br * (GP + 4), "modular elimination, one matrix per warp")
    # K4: 2^14 samples of dim_t = 1 (1.02 GB of float32 states)
    nb = 1 << 14
    idx = torch.randint(0, N * R, (nb,), device=dev, generator=torch.Generator(device=dev).manual_seed(0))
    store = env.DemoStore.from_tape(tape, slab, S, shift)
    t = timed(lambda: store.samples(idx, 1, replay_shift=shift), iters=5)
    report("tg_demo_sample_dm (K4, dim_t=1)", t, nb, "samples/s", nb * (4 * S ** 3 + GP + R // 2 * TP + 8 * 3 * S), "replay of ~R/2 records + float32 stores")
    t = timed(lambda: env.demo_samples(tape, slab, idx, S, 1, replay_shift=shift), iters=5)
    report("tg_demo_sample (K4, step-major, dim_t=1)", t, nb, "samples/s", nb * (4 * S ** 3 + GP + R // 2 * TP + 8 * 3 * S), "replay of ~R/2 records + float32 stores")
    f32 = torch.empty((nb, S, S, S), device=dev)
    sb = slab[:nb].contiguous()
    t = timed(lambda: env.expand_states(sb, S, out=f32), iters=10)
    report("tg_expand_f32", t, nb, "games/s", nb * (S * lay.row_pitch + 4 * S ** 3), "HBM")
    t = timed(lambda: env.pack_states(f32, S), iters=10)
    report("tg_pack_f32", t, nb, "games/s", nb * (GP + 4 * S ** 3), "HBM")

    print(f"{'kernel':44s} {'rate':>12s} {'unit':14s} {'GB/s':>7s} {'of copy':>8s}  bound")
    for name, rate, unit, bw, frac, bound in rows:
        print(f"{name:44s} {rate:12.4g} {unit:14s} {bw / 1e9:7.0f} {frac:8.2f}  {bound}")


if __name__ == "__main__":
    main()
