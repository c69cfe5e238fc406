"""The host-buffer path in its three slab formats: tg_step_host / tg_rollout_host (int8), their _i16 twins (int16 slabs)
and their _gf2 twins (bit slabs) at 4, 9, 16 and 25, from pinned host buffers, each next to its pinned-copy ceiling.

For every size and format: steps/s of the step (one PCIe round trip per step) and game-steps/s of the K = 23 rollout
(the slab crosses once per 23 steps), and the ceiling of each: the same bytes per call as plain cudaMemcpyAsync of
pinned memory in the same chunks, H2D and D2H on two streams at once, no kernel, measured in the same run.  A rate is
reported as a share of its ceiling.  Games are 9x9x9-style demos (tg_demo_gen_philox targets, R = 23) in every format:
the int16 slab holds the same targets (tg_demo_accumulate_i16) and the bit slab their residues (tg_pack_gf2).

2^20 games at 4 and 9, 2^17 at 16 and 2^15 at 25 (about 1 GiB per int16 slab at 16 and 25); 16 chunks per call.  Calls
return with the results in host memory, so each is timed with the host clock.

With --parent-lib PATH (the library of another build) the int8 rows are timed for both libraries, alternating parent,
this build, parent, this build, so that the difference can be read against the spread of the repeats.

Prints the card and its power limit first; run on the GPU:
    python scripts/time_host_formats.py [--parent-lib PATH] > profiles/host_formats_time.txt
"""
from __future__ import annotations

import argparse
import ctypes as C
import subprocess
import sys
import time
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from mat_mul_b200 import _lib, env  # noqa: E402

GAMES = {4: 1 << 20, 9: 1 << 20, 16: 1 << 17, 25: 1 << 15}
CHUNKS = 16
K = 23
SHIFT = 2
V5, P5 = (-2, -1, 0, 1, 2), (0.05, 0.10, 0.70, 0.10, 0.05)
HOST_FNS = ("tg_host_ctx_create", "tg_host_ctx_destroy", "tg_step_host", "tg_rollout_host")


def load_parent(path: str) -> C.CDLL:
    """another build's library, with the signatures of the int8 host entry points (unchanged since they were added)"""
    h = C.CDLL(path)
    for name in HOST_FNS:
        fn = getattr(h, name)
        fn.restype, fn.argtypes = _lib._SIGNATURES[name]
    return h


def copy_ceiling(dev, h2d: int, d2h: int, chunks: int, reps: int) -> float:
    """seconds per call of plain pinned copies of h2d bytes in and d2h bytes out, in `chunks` pieces on two streams"""
    hin, hout = torch.empty(h2d, dtype=torch.uint8, pin_memory=True), torch.empty(d2h, dtype=torch.uint8, pin_memory=True)
    din, dout = torch.empty(h2d, dtype=torch.uint8, device=dev), torch.empty(d2h, dtype=torch.uint8, device=dev)
    s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    ci, co = -(-h2d // chunks), -(-d2h // chunks)

    def one():
        for c in range(chunks):
            with torch.cuda.stream(s_in):
                din[c * ci:(c + 1) * ci].copy_(hin[c * ci:(c + 1) * ci], non_blocking=True)
            with torch.cuda.stream(s_out):
                hout[c * co:(c + 1) * co].copy_(dout[c * co:(c + 1) * co], non_blocking=True)

    one()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        one()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps


def timed(fn, reps: int) -> float:
    """seconds per call of a host-path call (it returns with the results in host memory)"""
    for _ in range(2):
        fn()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    return (time.perf_counter() - t0) / reps


def pinned_like(t: torch.Tensor) -> torch.Tensor:
    h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    h.copy_(t)
    return h


class Host:
    """pinned buffers of one size and format, and the two host calls on them through a library L"""

    def __init__(self, slab, tape_k, sfx: str):
        B = slab.shape[0]
        self.sfx, self.B = sfx, B
        self.slab, self.out = pinned_like(slab), torch.empty(slab.shape, dtype=slab.dtype, pin_memory=True)
        self.rec, self.tape = pinned_like(tape_k[K - 1]), pinned_like(tape_k.flip(0))
        self.flags = torch.empty(B, dtype=torch.uint8, pin_memory=True)
        self.nnz, self.steps = (torch.empty(B, dtype=torch.int32, pin_memory=True) for _ in range(2))
        self.slab_bytes = slab[0].numel() * slab.element_size()

    def calls(self, L, ctx):
        p = env._p
        step, roll = getattr(L, "tg_step_host" + self.sfx), getattr(L, "tg_rollout_host" + self.sfx)

        def one_step():
            _lib.check(step(ctx, p(self.slab), p(self.rec), p(self.out), p(self.flags), p(self.nnz), self.B, SHIFT), "step")

        def one_rollout():
            _lib.check(roll(ctx, p(self.slab), p(self.tape), K, p(self.out), p(self.flags), p(self.nnz), p(self.steps), self.B, SHIFT),
                       "rollout")
        return one_step, one_rollout


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", default=None, help="time the int8 rows for this library too, alternating")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "time_host_formats.py measures on the GPU"
    dev = torch.device("cuda:0")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print(f"card: {q[0] if q else torch.cuda.get_device_name(dev)}  (name, power limit, max SM clock)")
    print(f"pinned host buffers, {CHUNKS} chunks per call, {args.reps} timed calls after 2 warm-up calls; rollout K = {K}")
    print("bytes per game: step in = slab + TP, out = slab + 5; rollout in = slab + K*TP, out = slab + 9")
    L = _lib.lib()
    parent = load_parent(args.parent_lib) if args.parent_lib else None
    hdr = f"{'call':26s} {'S':>3s} {'games':>8s} {'B/game':>7s} {'rate':>11s} {'unit':14s} {'ceiling':>11s} {'share':>6s}"
    print(hdr, flush=True)
    ab = []
    for S in (4, 9, 16, 25):
        B, lay = GAMES[S], env.layout(S)
        chunk = B // CHUNKS
        tape, slab8, _ = env.make_synthetic_demos(B, K, S, V5, P5, SHIFT, seed=S, device=dev)
        slab16, _ = env.accumulate_demos16(tape, S, SHIFT)
        bits = env.pack_gf2(slab16, S)
        tape_k = tape.cpu()
        for fmt, slab in (("", slab8), ("_i16", slab16), ("_gf2", bits)):
            h = Host(slab.cpu(), tape_k, fmt)
            sb, tp = h.slab_bytes, lay.token_pitch
            ceil_step = copy_ceiling(dev, B * (sb + tp), B * (sb + 5), CHUNKS, args.reps)
            ceil_roll = copy_ceiling(dev, B * (sb + K * tp), B * (sb + 9), CHUNKS, args.reps)
            libs = [("", L)] if fmt or parent is None else [("parent ", parent), ("", L), ("parent ", parent), ("", L)]
            for tag, lib in libs:
                ctx = C.c_void_p()
                _lib.check(lib.tg_host_ctx_create(C.byref(ctx), 0, S, chunk), "tg_host_ctx_create")
                one_step, one_rollout = h.calls(lib, ctx)
                t_step, t_roll = timed(one_step, args.reps), timed(one_rollout, args.reps)
                lib.tg_host_ctx_destroy(ctx)
                name = tag + "tg_step_host" + fmt
                print(f"{name:26s} {S:3d} {B:8d} {2 * sb + tp + 5:7d} {B / t_step:11.4g} {'steps/s':14s} {B / ceil_step:11.4g} "
                      f"{ceil_step / t_step:6.3f}", flush=True)
                name = tag + "tg_rollout_host" + fmt
                print(f"{name:26s} {S:3d} {B:8d} {(2 * sb + K * tp + 9) // K:7d} {B * K / t_roll:11.4g} {'game-steps/s':14s} "
                      f"{B * K / ceil_roll:11.4g} {ceil_roll / t_roll:6.3f}", flush=True)
                if not fmt:
                    ab.append((S, tag or "new", B / t_step, B * K / t_roll))
            del h
        del tape, slab8, slab16, bits, tape_k
        torch.cuda.empty_cache()
    if parent is not None:
        print("\nint8 rows, this build / parent, per alternation pair (steps/s and game-steps/s)")
        for S in (4, 9, 16, 25):
            rows = [r for r in ab if r[0] == S]
            par, new = [r for r in rows if r[1] == "parent "], [r for r in rows if r[1] == "new"]
            ratios = [f"step {n[2] / p[2]:.3f} rollout {n[3] / p[3]:.3f}" for p, n in zip(par, new)]
            spread = [f"step {par[1][2] / par[0][2]:.3f} / {new[1][2] / new[0][2]:.3f}, rollout {par[1][3] / par[0][3]:.3f} / "
                      f"{new[1][3] / new[0][3]:.3f}"]
            print(f"S = {S:2d}: new/parent {'; '.join(ratios)}   repeat/first (parent / new): {spread[0]}")


if __name__ == "__main__":
    main()
