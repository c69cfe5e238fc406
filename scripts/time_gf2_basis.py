"""The change of basis over GF(2): tg_change_of_basis_gf2 at every size, the composition tg_unpack_gf2 ->
tg_change_of_basis -> tg_pack_gf2 at 4, 9 and 16 alternated with it in the same run, tg_change_of_basis_factors_gf2 and
tg_sample_invertible_gf2, with CUDA events, against a device-to-device copy measured in the same run.

Working sets are far above the 126 MB L2 (256-524 MB of bit slab per size) and every shape is warmed up before its timed
window.  Bytes are the traffic the formats imply, computed from the shapes: the transform reads and writes GB bytes per
game and reads its 12 S-byte triple (2 GB + 12 S = 80 / 332 / 1216 / 4300 bytes per game); the factors read and write
TP bytes per record; the sampler writes 12 S bytes per game.  Warp-instructions per game are counted from the SASS of
basis_gf2_kernel (cuobjdump): its body is unrolled, so the instructions of one pass of a CTA over its games, times the
CTA's warps, over its games; the issue bound is 4 warp-instructions per SM and cycle at the card's max SM clock.  Prints
the card and its power limit first; run on the GPU:  python scripts/time_gf2_basis.py > profiles/gf2_basis_time.txt
"""
from __future__ import annotations

import re
import shutil
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from mat_mul_b200 import _lib, env  # noqa: E402

GAMES = {4: 1 << 24, 9: 1 << 22, 16: 1 << 20, 25: 1 << 18}
R = 16  # records per game of the timed factor tapes


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


def sass_instructions() -> dict[int, int]:
    """S -> SASS instructions of basis_gf2_kernel<S> in the shipped library (empty without cuobjdump)."""
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    try:
        text = subprocess.run([exe, "-sass", str(_lib.LIB_PATH)], capture_output=True, text=True, check=True).stdout
    except (OSError, subprocess.CalledProcessError):
        return {}
    counts, cur = {}, None
    for line in text.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            k = re.search(r"basis_gf2_kernelILi(\d+)EE", m.group(1))
            cur = int(k.group(1)) if k else None
        elif cur is not None and re.match(r"\s*/\*[0-9a-f]{4}\*/\s+\S", line):
            counts[cur] = counts.get(cur, 0) + 1
    return counts


def main() -> None:
    assert torch.cuda.is_available(), "time_gf2_basis.py measures on the GPU"
    dev = torch.device("cuda:0")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print(f"card: {q[0] if q else torch.cuda.get_device_name(dev)}  (name, power limit, max SM clock)")
    clock_hz = float(re.search(r"(\d+) MHz", q[0]).group(1)) * 1e6 if q and "MHz" in q[0] else None
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    src = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
    dst = torch.empty_like(src)
    copy_bw = 2 * src.numel() / timed(lambda: dst.copy_(src))
    print(f"device-to-device copy of 1 GiB: {copy_bw / 1e9:.0f} GB/s (read + write)")
    del src, dst
    sass = sass_instructions()
    g = torch.Generator(device=dev).manual_seed(0)
    print(f"{'kernel':34s} {'S':>3s} {'games':>9s} {'rate':>11s} {'unit':10s} {'B/game':>7s} {'GB/s':>6s} {'of copy':>8s}")

    def row(name, S, games, t, n, unit, nbytes):
        print(f"{name:34s} {S:3d} {games:9d} {n / t:11.4g} {unit:10s} {nbytes / games:7.0f} {nbytes / t / 1e9:6.0f} "
              f"{nbytes / t / copy_bw:8.2f}", flush=True)

    for S, N in GAMES.items():
        lay, lg = env.layout(S), env.layout_gf2(S)
        GB, TP = lg.game_bytes, lay.token_pitch
        w = torch.randint(-(1 << 31), 1 << 31, (N, lg.game_words), generator=g, device=dev, dtype=torch.int64)
        bits = env.pack_gf2(env.unpack_gf2((w & 0xFFFFFFFF).to(torch.int32), S), S)  # clear the padding bits
        del w
        mats = env.sample_invertible_gf2(N, S, seed=1, p_nonzero=0.3)
        out = torch.empty_like(bits)
        native = lambda: env.change_of_basis_gf2(bits, mats, S, out=out)  # noqa: E731
        nbytes = N * (2 * GB + 12 * S)
        if S <= 16:  # the composition through the int8 slab, alternated with the native kernel
            m8 = env.sample_unimodular(N, S, seed=1, p_nonzero=0.3)
            s8, o8 = env.unpack_gf2(bits, S), torch.empty((N, lay.game_pitch), dtype=torch.int8, device=dev)

            def composed():
                env.unpack_gf2(bits, S)  # the unpacking the composition pays (its result is s8)
                env.change_of_basis(s8, m8, S, out=o8)
                return env.pack_gf2(o8, S)

            assert torch.equal(composed(), native())
            for rep in (1, 2):
                t = timed(native, iters=10)
                row(f"tg_change_of_basis_gf2 (rep {rep})", S, N, t, N, "games/s", nbytes)
                t = timed(composed, iters=3)
                row(f"unpack -> int8 basis -> pack ({rep})", S, N, t, N, "games/s", nbytes)
            del m8, s8, o8
        else:
            t = timed(native, iters=10)
            row("tg_change_of_basis_gf2", S, N, t, N, "games/s", nbytes)
        if S in sass:
            per_game = sass[S] * -(-(256 // S * S) // 32) / (256 // S)
            bound = f", issue bound {sms * 4 * clock_hz / per_game:.4g} games/s" if clock_hz else ""
            print(f"    basis_gf2_kernel<{S}>: {sass[S]} SASS instructions per thread and pass, {per_game:.0f} "
                  f"warp-instructions per game{bound}")
        Nf = N // 4
        tape = torch.randint(0, 256, (R, Nf, TP), generator=g, device=dev, dtype=torch.uint8)
        tape[..., 3 * S:] = 0
        tout = torch.empty_like(tape)
        L, st = _lib.lib(), env._stream()
        fac = lambda: L.tg_change_of_basis_factors_gf2(tape.data_ptr(), Nf * TP, 1, mats.data_ptr(), 1, tout.data_ptr(),  # noqa: E731
                                                      Nf * TP, 2, Nf, R, S, st)
        t = timed(fac, iters=5)
        row(f"factors_gf2 R={R}", S, Nf, t, Nf * R, "records/s", Nf * (2 * R * TP + 12 * S))
        t = timed(lambda: env.sample_invertible_gf2(N, S, seed=2, p_nonzero=0.3), iters=5)
        row("sample_invertible_gf2", S, N, t, N, "games/s", N * 12 * S)
        del bits, mats, out, tape, tout
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
