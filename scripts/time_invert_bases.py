"""Inverse triples: tg_invert_bases (over Z at 4, 9 and 16) and tg_invert_bases_gf2 (over GF(2) at 4, 9, 16 and 25) on
2^20 triples per size, with CUDA events, next to what the same N costs elsewhere in the change of basis: the sampler of the
bases (tg_sample_unimodular / tg_sample_invertible_gf2) and the tensor transform (tg_change_of_basis into an int8 slab /
tg_change_of_basis_gf2) of 2^20 zero games.  The inverse is paid once per basis, not per game step.

Every shape is warmed up before its timed window.  The integer triples are sampled at p_nonzero = 0.3, where about 1 % of
the 16x16 triples have no int8 inverse (they are flagged, at the same cost).  Prints the card and its power limit first;
run on the GPU:  python scripts/time_invert_bases.py > profiles/invert_bases_time.txt
"""
from __future__ import annotations

import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from mat_mul_b200 import env  # noqa: E402

N = 1 << 20


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
    assert torch.cuda.is_available(), "time_invert_bases.py measures on the GPU"
    dev = torch.device("cuda:0")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print(f"card: {q[0] if q else torch.cuda.get_device_name(dev)}  (name, power limit, max SM clock)")
    print(f"N = {N} triples (games) per row")
    print(f"{'call':34s} {'S':>3s} {'ms':>9s} {'triples/s':>11s} {'flagged':>8s}")

    def row(name, S, t, flagged=""):
        print(f"{name:34s} {S:3d} {t * 1e3:9.3f} {N / t:11.4g} {flagged:>8s}", flush=True)

    for S in (4, 9, 16):
        mats = env.sample_unimodular(N, S, seed=1, p_nonzero=0.3)
        inv = torch.empty_like(mats)
        _, flags = env.invert_bases(mats, out=inv)
        row("tg_invert_bases", S, timed(lambda: env.invert_bases(mats, out=inv)), f"{int((flags != 0).sum()) / N:.4f}")
        row("tg_sample_unimodular", S, timed(lambda: env.sample_unimodular(N, S, seed=2, p_nonzero=0.3)))
        slab = env.new_slab(N, S, dev)
        out = torch.empty_like(slab)
        row("tg_change_of_basis (int8 out)", S, timed(lambda: env.change_of_basis(slab, mats, S, out=out), iters=5))
        del mats, inv, slab, out
        torch.cuda.empty_cache()
    for S in (4, 9, 16, 25):
        mats = env.sample_invertible_gf2(N, S, seed=1, p_nonzero=0.3)
        inv = torch.empty_like(mats)
        _, flags = env.invert_bases_gf2(mats, out=inv)
        row("tg_invert_bases_gf2", S, timed(lambda: env.invert_bases_gf2(mats, out=inv)), f"{int((flags != 0).sum()) / N:.4f}")
        row("tg_sample_invertible_gf2", S, timed(lambda: env.sample_invertible_gf2(N, S, seed=2, p_nonzero=0.3)))
        bits = torch.zeros((N, env.layout_gf2(S).game_words), dtype=torch.int32, device=dev)
        out = torch.empty_like(bits)
        row("tg_change_of_basis_gf2", S, timed(lambda: env.change_of_basis_gf2(bits, mats, S, out=out), iters=5))
        del mats, inv, bits, out
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
