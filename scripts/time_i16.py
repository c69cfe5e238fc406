"""The int16 game path against the int8 one: K1 step, K8 leaf expansion, K2 rollout, K6 slice rank and K7 state key in
both formats side by side, with CUDA events, against a device-to-device copy measured in the same run.

The same games (entries in [-12, 12], so neither format flags them) and the same tapes (shift 2) go through both
formats.  Working sets are larger than the 126 MB L2, every shape is warmed up before its timed window, and the bytes
are the algorithmic traffic computed from the shapes (e = 1 or 2 bytes per entry): K1 reads and writes S^3 entries plus
3S tokens, flags and nnz (4 S^3 + 3S + 5 = 2948 B per int16 9x9x9 game-step).  Prints the card and its power limit
first; run on the GPU:  python scripts/time_i16.py > profiles/i16_time.txt
"""
from __future__ import annotations

import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from mat_mul_b200 import env  # noqa: E402

SHIFT = 2
GAMES = {4: 1 << 22, 9: 1 << 20, 16: 1 << 17, 25: 1 << 15}  # about 1 GB of int16 slab each


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
    assert torch.cuda.is_available(), "time_i16.py measures on the GPU"
    dev = torch.device("cuda:0")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print(f"card: {q[0] if q else torch.cuda.get_device_name(dev)}  (name, power limit, max SM clock)")
    src = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
    dst = torch.empty_like(src)
    copy_bw = 2 * src.numel() / timed(lambda: dst.copy_(src))
    print(f"device-to-device copy of 1 GiB: {copy_bw / 1e9:.0f} GB/s (read + write)")
    del src, dst
    g = torch.Generator(device=dev).manual_seed(0)
    print(f"{'kernel':34s} {'S':>3s} {'fmt':>5s} {'rate':>11s} {'unit':13s} {'GB/s':>6s} {'of copy':>8s}")

    for S, B in GAMES.items():
        lay = env.layout(S)
        GP, TP, S3 = lay.game_pitch, lay.token_pitch, S ** 3
        vals = torch.randint(-12, 13, (B, S, S, S), generator=g, device=dev, dtype=torch.float32)
        s8 = env.pack_states(vals, S)
        del vals
        s16 = s8.to(torch.int16)
        K, k = 16, 8
        toks = torch.randint(0, 2 * SHIFT + 1, (K * B, 3 * S), generator=g, device=dev)
        tape = env.pack_actions(toks, S).reshape(K, B, TP)
        del toks
        P = B // k
        tape_bk = tape[:k, :P].permute(1, 0, 2).contiguous()
        Br = B // 8

        def row(name, fmt, t, n, unit, nbytes):
            print(f"{name:34s} {S:3d} {fmt:>5s} {n / t:11.4g} {unit:13s} {nbytes / t / 1e9:6.0f} {nbytes / t / copy_bw:8.2f}", flush=True)

        for fmt, slab, e in (("int8", s8, 1), ("int16", s16, 2)):
            out = torch.empty_like(slab)
            t = timed(lambda: env.step_batch(slab, tape[0], S, SHIFT, out=out), iters=20)
            row("K1 step", fmt, t, B, "game-steps/s", B * (2 * e * S3 + 3 * S + 5))
        for fmt, slab, e in (("int8", s8, 1), ("int16", s16, 2)):
            parents = slab[:P].contiguous()
            t = timed(lambda: env.expand_children(parents, tape_bk, S, SHIFT), iters=5)
            row(f"K8 expand_children k={k}", fmt, t, P * k, "children/s", P * e * S3 + P * k * (e * S3 + 3 * S + 13))
        for fmt, slab, e in (("int8", s8, 1), ("int16", s16, 2)):
            out = torch.empty_like(slab)
            t = timed(lambda: env.rollout(slab, tape, S, SHIFT, out=out), iters=5)
            row(f"K2 rollout K={K}", fmt, t, B * K, "game-steps/s", 2 * B * e * S3 + K * B * 3 * S + 9 * B)
        for fmt, slab, e in (("int8", s8, 1), ("int16", s16, 2)):
            t = timed(lambda: env.state_keys(slab, S), iters=10)
            row("K7 state_key", fmt, t, B, "games/s", B * (e * S3 + 8))
        for fmt, slab, e in (("int8", s8, 1), ("int16", s16, 2)):
            sr = slab[:Br].contiguous()
            t = timed(lambda: env.slice_rank(sr, S), iters=3, warmup=1)
            row("K6 slice_rank", fmt, t, Br, "games/s", Br * (e * S3 + 4))
        assert torch.equal(env.step_batch(s8, tape[0], S, SHIFT)[0].to(torch.int16), env.step_batch(s16, tape[0], S, SHIFT)[0])
        del s8, s16, tape, tape_bk
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
