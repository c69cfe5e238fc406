"""The mod-2 training samples: tg_demo_sample_gf2 against the integer batcher tg_demo_sample_dm on an int8 store of the
same records and indices, and against that batcher followed by states.remainder_(2) (the composition it replaces), all
three alternated in one run with CUDA events; then tg_expand_f32_gf2 against tg_unpack_gf2 + tg_expand_f32.  The
device-to-device copy bandwidth is measured in the same run.

Stores are above the 126 MB L2 (R = 23 records per demo: 2^20 / 2^18 / 2^16 / 2^14 demos at 4 / 9 / 16 / 25, 290 to
450 MB of records and int8 targets), indices are uniform over the store, and every shape is warmed up before its timed
window.  Bytes are the traffic the formats imply, from the shapes and the sampled indices: a sample of the mod-2
batcher writes dim_t S^3 4 + 4 + 24 S + 4 bytes and reads GB + (R - a) TP + 8; the integer batcher reads GP target
bytes instead of GB; the remainder pass reads and writes the states once more.  Before timing, the states of (a) and
(c) are compared on the first 4096 samples.  Prints the card and its power limit first; run on the GPU:
    python scripts/time_gf2_samples.py > profiles/gf2_samples_time.txt
"""
from __future__ import annotations

import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from mat_mul_b200 import env  # noqa: E402

DEMOS = {4: 1 << 20, 9: 1 << 18, 16: 1 << 16, 25: 1 << 14}
GAMES = {4: 1 << 22, 9: 1 << 20, 16: 1 << 18, 25: 1 << 16}  # expansion: 0.7 to 4 GB of float32 out
R, SHIFT = 23, 2
V5, P5 = (-2, -1, 0, 1, 2), (0.05, 0.10, 0.70, 0.10, 0.05)


def timed(fn, iters: int, warmup: int = 1) -> float:
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
    assert torch.cuda.is_available(), "time_gf2_samples.py measures on the GPU"
    dev = torch.device("cuda:0")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print(f"card: {q[0] if q else torch.cuda.get_device_name(dev)}  (name, power limit, max SM clock)")
    src = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
    dst = torch.empty_like(src)
    copy_bw = 2 * src.numel() / timed(lambda: dst.copy_(src), 10)
    print(f"device-to-device copy of 1 GiB: {copy_bw / 1e9:.0f} GB/s (read + write)")
    del src, dst
    print(f"R = {R}, demo shift = replay_shift = {SHIFT}; (a) tg_demo_sample_gf2, (b) tg_demo_sample_dm on int8 targets, "
          f"(c) (b) + states.remainder_(2)")
    print(f"{'path':30s} {'S':>3s} {'nb':>7s} {'dim_t':>5s} {'samples/s':>11s} {'B/sample':>9s} {'GB/s':>6s} {'of copy':>8s} {'(b)/(a)':>8s} "
          f"{'(c)/(a)':>8s}")
    g = torch.Generator(device=dev).manual_seed(1)
    for S in (4, 9, 16, 25):
        lay, lay2 = env.layout(S), env.layout_gf2(S)
        N = DEMOS[S]
        tape, slab, _ = env.make_synthetic_demos(N, R, S, V5, P5, SHIFT, seed=S, device=dev)
        store8 = env.DemoStore.from_tape(tape, slab, S, SHIFT)
        store2 = env.DemoStore(store8.records, env.pack_gf2(slab, S), S, SHIFT)
        del tape, slab
        for nb in (1 << 16, 1 << 18):
            idx = torch.randint(0, N * R, (nb,), device=dev, generator=g)
            replayed = float((R - idx % R).sum()) * lay.token_pitch  # records a .. R-1 of every sample
            for dim_t in (1, 2, 4):
                small = idx[:4096]
                sa = store2.samples(small, dim_t, SHIFT)[0]
                sc = store8.samples(small, dim_t, SHIFT)[0].remainder_(2)
                assert torch.equal(sa, sc), (S, nb, dim_t)
                del sa, sc
                out = store2.samples(idx, dim_t, SHIFT)  # the output buffers, reused by all three paths

                def run_a():
                    env._call("tg_demo_sample_gf2", (store2.records,), env._p(store2.records), env._p(store2.targets), N, R, S, dim_t,
                              SHIFT, env._p(idx), nb, *map(env._p, out))

                def run_b():
                    env._call("tg_demo_sample_dm", (store8.records,), env._p(store8.records), env._p(store8.targets), 0, 127, N, R, S,
                              dim_t, SHIFT, env._p(idx), nb, *map(env._p, out))

                def run_c():
                    run_b()
                    out[0].remainder_(2)

                state_bytes = float(nb) * dim_t * S ** 3 * 4
                other = nb * (4 + 24 * S + 4 + 8)
                iters = 3 if state_bytes > 8e9 else 10
                ta, tb, tc = (timed(f, iters) for f in (run_a, run_b, run_c))
                ba = state_bytes + other + nb * lay2.game_bytes + replayed
                bb = state_bytes + other + nb * lay.game_pitch + replayed
                bc = bb + 2 * state_bytes
                for name, t, nbytes in (("(a) demo_sample_gf2", ta, ba), ("(b) demo_sample_dm int8", tb, bb),
                                        ("(c) (b) + remainder_(2)", tc, bc)):
                    ratios = f"{tb / ta:8.2f} {tc / ta:8.2f}" if name.startswith("(a)") else ""
                    print(f"{name:30s} {S:3d} {nb:7d} {dim_t:5d} {nb / t:11.4g} {nbytes / nb:9.0f} {nbytes / t / 1e9:6.0f} "
                          f"{nbytes / t / copy_bw:8.2f} {ratios}")
                del out
                torch.cuda.empty_cache()
        del store8, store2
        torch.cuda.empty_cache()
    print()
    print(f"{'path':34s} {'S':>3s} {'games':>8s} {'games/s':>11s} {'B/game':>7s} {'GB/s':>6s} {'of copy':>8s} {'speedup':>8s}")
    for S in (4, 9, 16, 25):
        B = GAMES[S]
        bits = torch.randint(-(1 << 31), 1 << 31, (B, env.layout_gf2(S).game_words), dtype=torch.int32, device=dev, generator=g)
        bits = env.pack_gf2(env.unpack_gf2(bits, S), S)  # zero padding bits and words
        f32 = torch.empty((B, S, S, S), dtype=torch.float32, device=dev)
        t1 = timed(lambda: env.expand_states(bits, S, out=f32), 10)
        t2 = timed(lambda: env.expand_states(env.unpack_gf2(bits, S), S, out=f32), 10)
        assert torch.equal(f32, env.expand_states(bits, S)), S
        b1 = B * (env.layout_gf2(S).game_bytes + 4 * S ** 3)
        b2 = b1 + 2 * B * env.layout(S).game_pitch
        print(f"{'tg_expand_f32_gf2':34s} {S:3d} {B:8d} {B / t1:11.4g} {b1 / B:7.0f} {b1 / t1 / 1e9:6.0f} {b1 / t1 / copy_bw:8.2f} {t2 / t1:8.2f}")
        print(f"{'tg_unpack_gf2 + tg_expand_f32':34s} {S:3d} {B:8d} {B / t2:11.4g} {b2 / B:7.0f} {b2 / t2 / 1e9:6.0f} {b2 / t2 / copy_bw:8.2f}")
        del bits, f32
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
