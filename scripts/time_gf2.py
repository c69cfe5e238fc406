"""The mod-2 game path on bit slabs: K1 step, K8 leaf expansion, K2 rollout, K7 state key and K6 slice rank at every size,
with CUDA events, against a device-to-device copy measured in the same run.

Working sets are far above the 126 MB L2 (2^24 games at 4x4x4: 256 MB of bit slab and 256 MB of records per step) and
every shape is warmed up before its timed window.  Bytes are the traffic the formats imply, computed from the shapes:
K1 reads and writes GB bytes per game and reads its TP-byte record, writes flags and nnz (GB = 16 / 112 / 512 / 2000,
TP = 16 / 32 / 48 / 80).  Records are random bytes (every byte is a token mod 2), so about 7/8 of the steps change a
game.  The int8 K1 at the same size is printed for comparison.  Prints the card and its power limit first; run on the
GPU:  python scripts/time_gf2.py > profiles/gf2_time.txt
"""
from __future__ import annotations

import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from mat_mul_b200 import env  # noqa: E402

SHIFT = 3
GAMES = {4: 1 << 24, 9: 1 << 22, 16: 1 << 20, 25: 1 << 18}  # 256-524 MB of bit slab each


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
    assert torch.cuda.is_available(), "time_gf2.py measures on the GPU"
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
    print(f"{'kernel':30s} {'S':>3s} {'games':>9s} {'rate':>11s} {'unit':13s} {'GB/s':>6s} {'of copy':>8s}")

    for S, B in GAMES.items():
        lay, lg = env.layout(S), env.layout_gf2(S)
        TP, GB = lay.token_pitch, lg.game_bytes
        K, k = 16, 8
        bits = torch.randint(-(1 << 31), 1 << 31, (B, lg.game_words), generator=g, device=dev, dtype=torch.int64)
        bits = env.pack_gf2(env.unpack_gf2((bits & 0xFFFFFFFF).to(torch.int32), S), S)  # clear the padding bits
        tape = torch.randint(0, 256, (K, B, TP), generator=g, device=dev, dtype=torch.uint8)
        tape[..., 3 * S:] = 0
        P = B // k
        tape_bk = tape[:k, :P].permute(1, 0, 2).contiguous()
        Br = B // 4

        def row(name, t, n, unit, nbytes, games=B):
            print(f"{name:30s} {S:3d} {games:9d} {n / t:11.4g} {unit:13s} {nbytes / t / 1e9:6.0f} {nbytes / t / copy_bw:8.2f}", flush=True)

        out = torch.empty_like(bits)
        t = timed(lambda: env.step_batch(bits, tape[0], S, SHIFT, out=out), iters=20)
        row("K1 step_gf2", t, B, "game-steps/s", B * (2 * GB + TP + 5))
        s8 = env.unpack_gf2(bits, S)
        o8 = torch.empty_like(s8)
        rec8 = tape[0] % 3  # tokens of the int8 alphabet for shift 1
        t = timed(lambda: env.step_batch(s8, rec8, S, 1, out=o8), iters=20)
        row("K1 step (int8, comparison)", t, B, "game-steps/s", B * (2 * lay.game_pitch + TP + 5))
        del s8, o8, rec8
        parents = bits[:P].contiguous()
        t = timed(lambda: env.expand_children(parents, tape_bk, S, SHIFT, with_keys=False), iters=5)
        row(f"K8 expand_children k={k}", t, P * k, "children/s", P * GB + P * k * (GB + TP + 5), P)
        t = timed(lambda: env.expand_children(parents, tape_bk, S, SHIFT), iters=5)
        row(f"K8 expand_children k={k} keys", t, P * k, "children/s", P * GB + P * k * (GB + TP + 13), P)
        t = timed(lambda: env.rollout(bits, tape, S, SHIFT, out=out), iters=5)
        row(f"K2 rollout K={K}", t, B * K, "game-steps/s", 2 * B * GB + K * B * TP + 9 * B)
        t = timed(lambda: env.replay(bits, tape, S, SHIFT, out=out), iters=5)
        row(f"K2 replay K={K}", t, B * K, "game-steps/s", 2 * B * GB + K * B * TP + 5 * B)
        t = timed(lambda: env.state_keys(bits, S), iters=10)
        row("K7 state_key_gf2", t, B, "games/s", B * (GB + 8))
        sr = bits[:Br].contiguous()
        t = timed(lambda: env.slice_rank(sr, S), iters=5)
        row("K6 slice_rank_gf2", t, Br, "games/s", Br * (GB + 4), Br)
        del bits, tape, tape_bk, parents, out, sr
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
