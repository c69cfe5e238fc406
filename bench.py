#!/usr/bin/env python
"""Headline benchmark of the TensorGame hot path on B200.

Workload (BASELINE.json configs[1]): 3x3 matmul tensor (9x9x9), 2^20 parallel games per GPU, coefficients {-2..2}.
BASELINE.json's metric has two halves, both measured here on that configuration:
  --metric steps (default)  env steps/s: one "step" = one tg_step launch over the whole batch (every game makes one
                            transition);
  --metric demos            synthetic demos/s: one "step" = one tg_demo_gen_philox launch generating the whole batch.
The default line also carries the other half as a first-class block (`demos`, with its own roofline, cpu_baseline and
e2e).  See DESIGN.md "Measurement".

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--metric steps|demos] [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  For N>1 launch with torch.distributed.run.

--dump-outputs DIR writes what the last timed step returned, as DIR/<name>.npy in float32: the step's (slab, flags, nnz)
(--metric steps) or the generator's (tape, slab, flags) (--metric demos).  The inputs are seeded, so the same arguments
give the same arrays on every run and two builds can be compared file by file.  Arrays larger than the dump budget keep
the games of one fixed, seeded sample, the same games in every array.  At N > 1 rank 0 writes its shard, which holds the
same games as a one-GPU run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

STEP_BYTES = {4: 145, 9: 1490, 16: 8245}  # SURVEY.md 8(d): 2*S^3 + 3S + 1 + 4 per env step
DEMO_R = {4: 7, 9: 23, 16: 49}
FALLBACK_HBM_GBS = 6650.0  # B200_PROFILING.md fallback
VALUES5, PROBS5 = (-2, -1, 0, 1, 2), (0.05, 0.10, 0.70, 0.10, 0.05)  # P(0) = 0.7 as in the reference (datasets.py:31)
VALUES3, PROBS3 = (-1, 0, 1), (0.15, 0.7, 0.15)                      # the reference's defaults (datasets.py:30-31)
REF_DIR = ROOT / "baseline" / "_ref"  # verbatim copy of the reference's scripts (scripts/install_ref.sh), if installed
DUMP_BYTES = 60_000_000  # --dump-outputs budget: under 64 MB with the .npy headers
DUMP_NAMES = ("slab", "flags", "nnz", "tape")  # the files --dump-outputs writes: steps (slab, flags, nnz), demos (tape, slab, flags)


def demo_bytes(S: int, R: int) -> int:
    """SURVEY.md 8(d): S^3 + R*3S bytes written per synthetic demo."""
    return S ** 3 + R * 3 * S


def parse() -> argparse.Namespace:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--metric", default="steps", choices=["steps", "demos"])
    ap.add_argument("--size", type=int, default=9, choices=[4, 9, 16], help="dim_3d S")
    ap.add_argument("--games", type=int, default=1 << 20, help="games per GPU")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--ctas-per-sm", type=int, default=0, help="tuning sweep only (TG_TUNING=1 build)")
    ap.add_argument("--variant", type=int, default=0, help="tuning sweep only (TG_TUNING=1 build)")
    ap.add_argument("--dump-outputs", type=Path, default=None, metavar="DIR",
                    help="write the outputs of the last timed step to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours (the reference arm times CPU code)")
    return args


def workload_config(metric: str, S: int, B: int, shift: int, world: int) -> dict:
    """The `config` object; both arms print exactly this for the same flags."""
    rp = (S * S + 3) & ~3
    gp, tp = (S * rp + 15) & ~15, (3 * S + 15) & ~15
    if metric == "steps":
        touched = (2 * gp + tp) * B
        what = f"tensorgame step {S}x{S}x{S}, 2^{B.bit_length() - 1} games per GPU, coefficients -2..2"
    else:
        touched = (gp + DEMO_R[S] * tp) * B
        what = f"synthetic demos {S}x{S}x{S} rank {DEMO_R[S]}, 2^{B.bit_length() - 1} demos per GPU, coefficients -2..2"
    return {"workload": what, "games_per_gpu": B, "size": S, "shift": shift,
            "sharding": f"game index, {world} rank(s), no data-path collective",
            "l2": f"inputs larger than L2 ({touched >> 20} MiB touched per step)"}


def hbm_peak() -> tuple[float, str]:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            self.path = tempfile.NamedTemporaryFile(prefix="clocks_", suffix=".csv", delete=False).name
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.index)],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        self.proc.wait()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        os.unlink(self.path)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def _time_ms(fn, iters: int, torch) -> float:
    for _ in range(3):  # first launches carry host-side module-load latency
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


# ------------------------------------------------------------------------------------------------ --dump-outputs
def sample_outputs(outputs: dict, B: int) -> dict:
    """Host float32 copies of device outputs, each given as (tensor, dimension indexing the B games).  Over the
    DUMP_BYTES budget every array keeps the same fixed, seeded, sorted sample of games."""
    import numpy as np
    import torch

    per_game = sum(t.numel() // B for t, _ in outputs.values()) * 4
    n = min(B, DUMP_BYTES // per_game)
    idx = None if n == B else torch.from_numpy(np.sort(np.random.default_rng(0).choice(B, n, replace=False)))
    host = {}
    for name, (t, dim) in outputs.items():
        if idx is not None:
            t = t.index_select(dim, idx.to(t.device))
        host[name] = t.cpu().numpy().astype(np.float32)
    return host


def write_outputs(out_dir: Path, host: dict) -> None:
    """DIR/<name>.npy for every array; a file another run left under one of the names either metric writes is removed
    first, so that DIR holds exactly this run's outputs."""
    import numpy as np

    assert set(host) <= set(DUMP_NAMES), sorted(host)
    out_dir.mkdir(parents=True, exist_ok=True)
    for name in DUMP_NAMES:
        (out_dir / f"{name}.npy").unlink(missing_ok=True)
    for name, a in host.items():
        np.save(out_dir / f"{name}.npy", a)


# ------------------------------------------------------------------------------------------------ CPU legs
def cpu_step_port(S: int, shift: int, seconds: float):
    """The oracle's C port of training.py:253-266 on the reference's dtypes (float32 residuals, int64 tokens), OpenMP
    over games on every host core.  Returns (steps/s, cores, sample description) from a bounded sample."""
    import numpy as np

    from oracle import tg_oracle as orc

    cores = orc.use_all_threads()  # torchrun exports OMP_NUM_THREADS=1 to its workers: the CPU arm uses every core regardless
    Bs = 1 << 16
    rng = np.random.default_rng(0)
    T = (rng.integers(-2, 3, (Bs, S, S, S)) * (rng.random((Bs, S, S, S)) < 0.3)).astype(np.float32)
    tok = rng.integers(0, 2 * shift + 1, (Bs, 3 * S)).astype(np.int64)
    tok[rng.random((Bs, 3 * S)) < 0.6] = shift
    out = np.empty_like(T); flags = np.empty(Bs, np.uint8); nnz = np.empty(Bs, np.int32)
    orc.step_batch_f32(T, tok, shift, out, flags, nnz)  # warm
    t0 = time.perf_counter()
    orc.step_batch_f32(T, tok, shift, out, flags, nnz)
    one = time.perf_counter() - t0
    reps = max(1, min(20000, int(seconds / max(one, 1e-6))))
    t0 = time.perf_counter()
    for _ in range(reps):
        orc.step_batch_f32(T, tok, shift, out, flags, nnz)
    dt = time.perf_counter() - t0
    return reps * Bs / dt, cores, (f"{reps} passes over {Bs} games of {S}x{S}x{S} ({dt:.1f} s), C port of training.py:253-266 on "
                                   "float32/int64, OpenMP over games")


def _import_reference():
    """The reference's own utils module from baseline/_ref (None if not installed)."""
    if not (REF_DIR / "utils.py").exists():
        return None
    import importlib.util

    spec = importlib.util.spec_from_file_location("_tg_reference_utils", REF_DIR / "utils.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def cpu_step_reference(S: int, seconds: float, n_samples: int = 8):
    """The reference's own batched step (training.py:253-267: tokens - 2, utils.uvw_to_tensor, head - action tensor,
    history shift, nnz per group, min over samples) in torch on every host core.  None if baseline/_ref is absent."""
    ref = _import_reference()
    if ref is None:
        return None
    import torch

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    B, T = 1 << 13, 2
    g = torch.Generator().manual_seed(0)
    state = (torch.randint(-2, 3, (B, T, S, S, S), generator=g) * (torch.rand((B, T, S, S, S), generator=g) < 0.3)).float()
    aa = torch.randint(0, 5, (B, 1, 3 * S), generator=g)

    def step(state_batch):
        uu, vv, ww = torch.split(aa.squeeze() - 2, S, dim=-1)            # training.py:253
        action_tensor = ref.uvw_to_tensor((uu, vv, ww))                   # :254
        new_head = state_batch[:, 0] - action_tensor                      # :255
        new_state = torch.cat((new_head.unsqueeze(1), state_batch), dim=1)[:, :-1]  # :257-258
        rank_ubs = torch.sum(new_head.view(-1, n_samples, S, S, S) != 0, dim=(-1, -2, -3), dtype=torch.int32)  # :259-266
        return new_state, rank_ubs.min(dim=1)                             # :267

    step(state)
    t0 = time.perf_counter()
    step(state)
    one = time.perf_counter() - t0
    reps = max(1, min(2000, int(seconds / max(one, 1e-6))))
    t0 = time.perf_counter()
    for _ in range(reps):
        state, _ = step(state)
    dt = time.perf_counter() - t0
    return reps * B / dt, cores, (f"{reps} passes over {B} games of {S}x{S}x{S} ({dt:.1f} s): the reference's own expression "
                                  f"training.py:253-267 with baseline/_ref/utils.uvw_to_tensor, torch CPU, {cores} threads")


def cpu_demo_port(S: int, R: int, shift: int, values, probs, seconds: float):
    """The oracle's C restatement of the demo generator (same Philox contract as the kernel), OpenMP over demos."""
    from oracle import tg_oracle as orc

    cores = orc.use_all_threads()
    n = 1 << 12
    orc.demos_philox(1, 0, n, values, probs, R, S, shift)
    t0 = time.perf_counter()
    orc.demos_philox(1, 0, n, values, probs, R, S, shift)
    one = time.perf_counter() - t0
    reps = max(1, min(20000, int(seconds / max(one, 1e-6))))
    t0 = time.perf_counter()
    for i in range(reps):
        orc.demos_philox(1, i * n, n, values, probs, R, S, shift)
    dt = time.perf_counter() - t0
    return reps * n / dt, cores, f"{reps} batches of {n} demos {S}x{S}x{S} rank {R} ({dt:.1f} s), C port of utils.py:203-233, OpenMP over demos"


def cpu_demo_reference(S: int, R: int, shift: int, values, probs, seconds: float):
    """The reference's own create_synthetic_demo loop (utils.py:203-233; single Python thread, as it has no parallel
    path).  None if baseline/_ref is absent."""
    ref = _import_reference()
    if ref is None:
        return None
    import torch

    v, p = torch.tensor(values), torch.tensor(probs)
    torch.manual_seed(0)
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        ref.create_synthetic_demo(v, p, R, S, shift)
        n += 1
    dt = time.perf_counter() - t0
    return n / dt, 1, f"{n} calls of baseline/_ref/utils.create_synthetic_demo ({dt:.1f} s), {S}x{S}x{S} rank {R}, one Python thread"


# ------------------------------------------------------------------------------------------------ reference arm
def run_reference(args) -> None:
    """--impl reference: rank 0 times the reference's CPU implementation of the path; other ranks exit.  With
    baseline/_ref installed the value is the reference's OWN code (kind "reference"); the C/OpenMP port of the same
    expression (a much stronger baseline) is reported beside it, and is the value when baseline/_ref is absent."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    S, shift = args.size, 2
    budget = 4.0  # seconds of CPU work per timed step
    if args.metric == "steps":
        port = lambda s: cpu_step_port(S, shift, s)          # noqa: E731
        real = lambda s: cpu_step_reference(S, s)            # noqa: E731
        metric, unit, dtype = "env_steps_per_sec", "steps/s", "f32"
    else:
        R = DEMO_R[S]
        port = lambda s: cpu_demo_port(S, R, shift, VALUES5, PROBS5, s)       # noqa: E731
        real = lambda s: cpu_demo_reference(S, R, shift, VALUES5, PROBS5, s)  # noqa: E731
        metric, unit, dtype = "synthetic_demos_per_sec", "demos/s", "f32"
    have_ref = real(0.2) is not None
    leg = real if have_ref else port
    for _ in range(args.warmup):
        leg(0.2)
    t0 = time.perf_counter()
    vals = [leg(budget) for _ in range(max(args.steps, 1))]
    dt = time.perf_counter() - t0
    value = sum(v[0] for v in vals) / len(vals)
    cores, sample = vals[-1][1], vals[-1][2]
    pv = port(budget)
    kind = "reference" if have_ref else "port"
    line = {
        "impl": "reference", "metric": metric, "value": value, "unit": unit, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / max(args.steps, 1) * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": dtype, "data": "synthetic",
        "config": workload_config(args.metric, S, args.games, shift, args.gpus),
        "cpu_baseline": {"value": value, "unit": unit, "cores": cores, "kind": kind,
                         "sample": f"each step: {sample}"},
        "port": {"value": pv[0], "unit": unit, "cores": pv[1], "kind": "port", "sample": pv[2]},
        "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ e2e helpers
def copy_ceiling(torch, dev, h2d_bytes: int, d2h_bytes: int, chunks: int, reps: int, barrier=None) -> float:
    """Raw bidirectional pinned-copy ceiling of this host<->GPU path: the bytes one e2e step moves, as plain async
    copies in the same chunking on two streams (H2D and D2H concurrently), no kernel.  Returns seconds per step.
    `barrier` is called after the buffers exist and the copies are warm, so that at N > 1 every rank's timed copies
    run while all the others' do (allocation / pinning takes a different time on every rank)."""
    hin = torch.empty(h2d_bytes, dtype=torch.uint8).pin_memory()
    hout = torch.empty(d2h_bytes, dtype=torch.uint8).pin_memory()
    din = torch.empty(h2d_bytes, dtype=torch.uint8, device=dev)
    dout = torch.empty(d2h_bytes, dtype=torch.uint8, device=dev)
    s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    ci, co = -(-h2d_bytes // chunks), -(-d2h_bytes // chunks)

    def one():
        for c in range(chunks):
            with torch.cuda.stream(s_in):
                din[c * ci:(c + 1) * ci].copy_(hin[c * ci:(c + 1) * ci], non_blocking=True)
            with torch.cuda.stream(s_out):
                hout[c * co:(c + 1) * co].copy_(dout[c * co:(c + 1) * co], non_blocking=True)

    one()
    torch.cuda.synchronize()
    if barrier is not None:
        barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        one()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps


def max_over_ranks(x: float, torch, dist, dev, world: int) -> float:
    t = torch.tensor([x], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


# ------------------------------------------------------------------------------------------------ demos block
def measure_demos(env, torch, dist, dev, S, B, R, values, probs, shift, world, rank, local, barrier, K, with_e2e, with_cpu,
                  tape=None, slab=None, dump=False) -> dict:
    """Synthetic demos/s (the other half of BASELINE.json's metric) as a first-class measurement: device-timed value,
    roofline of the generator kernel, end to end into pinned host memory (tg_demo_gen_host), CPU baselines.  With
    `dump`, out["outputs"] holds host copies of the last timed launch's (tape, slab, flags)."""
    lay = env.layout(S)
    peak, peak_kind = hbm_peak()
    if tape is None:
        tape = torch.empty((R, B, lay.token_pitch), dtype=torch.uint8, device=dev)
    if slab is None:
        slab = torch.empty((B, lay.game_pitch), dtype=torch.int8, device=dev)
    gen = lambda i: env.make_synthetic_demos(B, R, S, values, probs, shift, seed=0xD0 + i, first_demo=rank * B, device=dev,  # noqa: E731
                                             tape=tape, slab=slab)
    for i in range(3):
        gen(i)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        _, _, dflags = gen(i)
    e1.record()
    barrier()
    outputs = sample_outputs({"tape": (tape, 1), "slab": (slab, 0), "flags": (dflags, 0)}, B) if dump else None
    ms = max_over_ranks(e0.elapsed_time(e1) / K, torch, dist, dev, world)
    algo = demo_bytes(S, R)
    achieved = B * algo / (ms * 1e-3) / 1e9
    out = {"metric": "synthetic_demos_per_sec", "value": world * B / ms * 1e3, "unit": "demos/s", "ms_per_step": ms, "steps": K,
           "demos_per_gpu": B, "size": S, "R": R, "dtype": "int8", "gpu_launches": K * world,
           "flagged": int((dflags != 0).sum().item()),
           "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                        "traffic": None, "peak_kind": peak_kind, "kernel": "tg::demo_kernel",
                        "algorithmic_bytes_per_demo": algo, "moved_bytes_per_demo": lay.game_pitch + R * lay.token_pitch + 1,
                        "note": "write-only; the kernel is bound by INT-pipe issue slots (Philox draws + packed rank-1 "
                                "accumulation), reported against the HBM roofline as SURVEY 8(d) asks"}}
    if with_e2e:
        h_tape = torch.empty((R, B, lay.token_pitch), dtype=torch.uint8).pin_memory()
        h_slab = torch.empty((B, lay.game_pitch), dtype=torch.int8).pin_memory()
        h_flags = torch.empty(B, dtype=torch.uint8).pin_memory()
        hs = env.HostStepper(S, local, chunk=1 << 16)
        hs.make_demos(h_tape, h_slab, h_flags, shift, values, probs, seed=0xD0, first_demo=rank * B)
        barrier()
        Ke = max(2, min(K, 5))
        t0 = time.perf_counter()
        for i in range(Ke):
            hs.make_demos(h_tape, h_slab, h_flags, shift, values, probs, seed=0xD0 + i, first_demo=rank * B)
        dt = max_over_ranks((time.perf_counter() - t0) / Ke, torch, dist, dev, world)
        hs.close()
        d2h = B * (lay.game_pitch + R * lay.token_pitch + 1)
        ceil_s = max_over_ranks(copy_ceiling(torch, dev, 16, d2h, 16, Ke, barrier), torch, dist, dev, world)
        # the host copy equals the device result of the same seed (checked on a slice, outside the timed region)
        gen(Ke - 1)
        same = bool(torch.equal(h_slab[:4096], slab[:4096].cpu()) and torch.equal(h_tape[:, :4096], tape[:, :4096].cpu()))
        out["e2e"] = {"value": world * B / dt, "unit": "demos/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": d2h, "steps": Ke,
                      "api": "tg_demo_gen_host (C ABI, pinned host buffers, 64Ki-demo chunks through dedicated kernel / D2H streams chained by events)",
                      "ceiling_gbs": d2h / ceil_s / 1e9, "frac_of_ceiling": (d2h / dt) / (d2h / ceil_s), "host_equals_device": same}
        del h_tape, h_slab
    if with_cpu and world == 1:
        v, cores, sample = cpu_demo_port(S, R, shift, values, probs, 6.0)
        out["cpu_baseline"] = {"value": v, "unit": "demos/s", "cores": cores, "kind": "port", "sample": sample}
        real = cpu_demo_reference(S, R, shift, values, probs, 4.0)
        if real is not None:
            out["cpu_reference"] = {"value": real[0], "unit": "demos/s", "cores": real[1], "kind": "reference", "sample": real[2]}
    if dump:
        out["outputs"] = outputs
    return out


# ------------------------------------------------------------------------------------------------ extras
def measure_extras(env, dev, S, shift, slab, tape3, R, values, probs, world, rank, barrier) -> dict:
    """The other kernels of the path on the same games (per-GPU numbers, CUDA events, a few launches each): fused
    rollout, change of basis at SURVEY 8(d)'s configuration (int16 out, p_nonzero 0.3), training-sample batcher,
    leaf expansion, rank reward; the 4x4x4 and 16x16x16 sizes; at N > 1 the collectives of the path."""
    import torch

    from mat_mul_b200 import dist as tgd

    B = slab.shape[0]
    lay = env.layout(S)
    peak, _ = hbm_peak()
    out = {"per_gpu": True, "n_gpus": world}
    s2 = torch.empty_like(slab)
    ms = _time_ms(lambda: env.accumulate_demos(tape3, S, shift, slab=s2), 3, torch)
    out["demo_accumulate"] = {"value": B / ms * 1e3, "unit": "demos/s", "ms": ms}
    rev = tape3.flip(0).contiguous()
    ms = _time_ms(lambda: env.rollout(slab, rev, S, shift, out=s2), 3, torch)
    algo = 2 * S ** 3 + R * 3 * S + 8
    out["rollout"] = {"metric": "env_steps_per_sec (fused K-step rollout)", "value": B * R / ms * 1e3, "games_per_sec": B / ms * 1e3,
                      "K": R, "ms": ms, "hbm_frac": B * algo / (ms * 1e-3) / 1e9 / peak}
    del rev, s2

    def basis_block(Sx, slab_x, n, p_nz):
        """Change of basis at SURVEY 8(d)'s configuration: one unimodular (A, B, C) per game, off-diagonal entries
        non-zero with probability p_nz (config 3: 0.3), int8 in, int16 out: S^3 + 3S^2 + 2S^3 bytes per game."""
        mats = env.sample_unimodular(n, Sx, seed=3, p_nonzero=p_nz, device=dev)
        o16 = torch.empty((n, env.layout(Sx).game_pitch), dtype=torch.int16, device=dev)
        res = {}
        ms16 = _time_ms(lambda: env.change_of_basis(slab_x[:n], mats, Sx, out=o16), 5, torch)
        _, fl, stats = env.change_of_basis(slab_x[:n], mats, Sx, out=o16, return_path_stats=True)
        by = Sx ** 3 + 3 * Sx * Sx + 2 * Sx ** 3
        res["int16_out"] = {"value": n / ms16 * 1e3, "unit": "games/s", "ms": ms16, "games": n, "p_nonzero": p_nz,
                            "bytes_per_game": by, "hbm_frac": n * by / (ms16 * 1e-3) / 1e9 / peak,
                            "int_ops_per_game": 6 * Sx ** 4, "paths": stats,
                            "out_of_int16": int(((fl & env.FLAG_RANGE) != 0).sum().item())}
        o8 = torch.empty((n, env.layout(Sx).game_pitch), dtype=torch.int8, device=dev)
        ms8 = _time_ms(lambda: env.change_of_basis(slab_x[:n], mats, Sx, out=o8), 5, torch)
        _, fl8 = env.change_of_basis(slab_x[:n], mats, Sx, out=o8)
        by8 = 2 * Sx ** 3 + 3 * Sx * Sx
        res["int8_out"] = {"value": n / ms8 * 1e3, "unit": "games/s", "ms": ms8, "bytes_per_game": by8,
                           "hbm_frac": n * by8 / (ms8 * 1e-3) / 1e9 / peak,
                           "beyond_int8_zone": int(((fl8 & env.FLAG_RANGE) != 0).sum().item())}
        return res, mats

    nb = min(B, 1 << 18)
    out["change_of_basis"], _ = basis_block(S, slab, nb, 0.3)
    idx = torch.randint(0, B * R, (1 << 16,), device=dev)
    store = env.DemoStore.from_tape(tape3, slab, S, shift)  # demo-major action records next to the step-major tape
    ms = _time_ms(lambda: store.samples(idx, 2, replay_shift=shift), 10, torch)
    out["demo_sample"] = {"value": idx.numel() / ms * 1e3, "unit": "samples/s", "ms": ms, "dim_t": 2, "samples": idx.numel(),
                          "hbm_frac": idx.numel() * (2 * S ** 3 * 4) / (ms * 1e-3) / 1e9 / peak}
    # the same batcher on a batch four times as large (the tail of the persistent grid weighs less) and with four state slots
    idx4 = torch.randint(0, B * R, (1 << 18,), device=dev)
    for key, ii, T in (("batch_2e18", idx4, 2), ("dim_t_4", idx, 4)):
        ms = _time_ms(lambda: store.samples(ii, T, replay_shift=shift), 5, torch)
        out["demo_sample"][key] = {"value": ii.numel() / ms * 1e3, "ms": ms, "dim_t": T, "samples": ii.numel(),
                                   "hbm_frac": ii.numel() * (T * S ** 3 * 4) / (ms * 1e-3) / 1e9 / peak}
    del idx4
    del store
    # batched leaf expansion (K8): k = 8 candidate actions per state, children + flags + nnz (+ keys)
    nbp = min(B, 1 << 17)
    tape_bk = tape3[:8, :nbp].permute(1, 0, 2).contiguous()
    kk = tape_bk.shape[1]
    moved = lay.game_pitch * (1 + 1 / kk) + lay.token_pitch + 5
    ms = _time_ms(lambda: env.expand_children(slab[:nbp], tape_bk, S, shift, with_keys=False), 3, torch)
    ms_k = _time_ms(lambda: env.expand_children(slab[:nbp], tape_bk, S, shift, with_keys=True), 3, torch)
    out["expand_children"] = {"value": nbp * kk / ms * 1e3, "unit": "children/s", "k": kk, "ms": ms,
                              "hbm_frac": nbp * kk * moved / (ms * 1e-3) / 1e9 / peak,
                              "with_state_keys": {"value": nbp * kk / ms_k * 1e3, "ms": ms_k}}
    del tape_bk
    ms = _time_ms(lambda: env.slice_rank(slab[:nbp], S), 3, torch)
    out["slice_rank"] = {"value": nbp / ms * 1e3, "unit": "games/s", "ms": ms,
                         "bound": "ALU (modular elimination, S^3/3 multiply-adds per slice); reads S^3 bytes per game",
                         "hbm_frac": nbp * S ** 3 / (ms * 1e-3) / 1e9 / peak}
    if S == 9:
        # BASELINE.json quotes the metric at 4x4x4 too: env steps on 2^22 games of the 2x2 matmul size
        # (reference defaults: coefficients {-1,0,1}, P(0) = 0.7, R = 7, shift = 1); demos/s at 4x4x4 is in `demos_4x4x4`
        S4, R4, B4 = 4, 7, 1 << 22
        t4, s4, _ = env.make_synthetic_demos(B4, R4, S4, VALUES3, PROBS3, 1, seed=2, device=dev)
        o4, f4, n4 = torch.empty_like(s4), torch.empty(B4, dtype=torch.uint8, device=dev), torch.empty(B4, dtype=torch.int32, device=dev)
        ms_step = _time_ms(lambda: env.step_batch(s4, t4[R4 - 1], S4, 1, out=o4, flags=f4, nnz=n4), 10, torch)
        out["size_4x4x4"] = {"games": B4, "env_steps_per_sec": B4 / ms_step * 1e3, "step_ms": ms_step,
                             "step_hbm_frac": B4 * STEP_BYTES[4] / (ms_step * 1e-3) / 1e9 / peak}
        # change of basis at 4x4x4: one thread per game, exact int32 in registers (csrc/tg_basis.cu basis4_thread_kernel)
        out["size_4x4x4"]["change_of_basis"], _ = basis_block(S4, s4, 1 << 20, 0.3)
        # sample batcher at 4x4x4 (the reference's default size): four threads per sample, rows in registers
        st4 = env.DemoStore.from_tape(t4, s4, S4, 1)
        i4 = torch.randint(0, B4 * R4, (1 << 20,), device=dev)
        ms_s4 = _time_ms(lambda: st4.samples(i4, 2, replay_shift=1), 5, torch)
        out["size_4x4x4"]["demo_sample"] = {"value": i4.numel() / ms_s4 * 1e3, "unit": "samples/s", "ms": ms_s4, "dim_t": 2,
                                            "samples": i4.numel(),
                                            "hbm_frac": i4.numel() * (2 * S4 ** 3 * 4) / (ms_s4 * 1e-3) / 1e9 / peak}
        del st4, i4
        torch.cuda.empty_cache()  # the blocks below allocate 0.5 GB outputs of other sizes: keep the allocator's pools apart
        # fused rollout at 4x4x4: one thread per game, the game in registers for all K steps
        rev4 = t4.flip(0).contiguous()
        ms_r4 = _time_ms(lambda: env.rollout(s4, rev4, S4, 1, out=o4), 5, torch)
        out["size_4x4x4"]["rollout"] = {"value": B4 * R4 / ms_r4 * 1e3, "unit": "game-steps/s", "K": R4, "ms": ms_r4,
                                        "hbm_frac": B4 * (2 * S4 ** 3 + R4 * 3 * S4 + 8) / (ms_r4 * 1e-3) / 1e9 / peak}
        del rev4
        # batched leaf expansion at 4x4x4: four threads per parent, rows in registers, k = 7 candidate actions per state
        nb4 = 1 << 20
        tb4 = t4[:, :nb4].permute(1, 0, 2).contiguous()
        k4 = tb4.shape[1]
        moved4 = 64 * (1 + 1 / k4) + 16 + 5
        ms_e4 = _time_ms(lambda: env.expand_children(s4[:nb4], tb4, S4, 1, with_keys=False), 5, torch)
        ms_e4k = _time_ms(lambda: env.expand_children(s4[:nb4], tb4, S4, 1, with_keys=True), 5, torch)
        out["size_4x4x4"]["expand_children"] = {"value": nb4 * k4 / ms_e4 * 1e3, "unit": "children/s", "k": k4, "ms": ms_e4,
                                                "hbm_frac": nb4 * k4 * moved4 / (ms_e4 * 1e-3) / 1e9 / peak,
                                                "with_state_keys": {"value": nb4 * k4 / ms_e4k * 1e3, "ms": ms_e4k,
                                                                    "hbm_frac": nb4 * k4 * (moved4 + 8) / (ms_e4k * 1e-3) / 1e9 / peak}}
        del tb4
        del t4, s4, o4
        # BASELINE.json configs[2]: 16x16x16 demos (rank <= 49) followed by the change-of-basis augmentation, one
        # (A, B, C) triple per demo -- the one contraction that runs on the tensor cores (csrc/tg_basis_mma.cu)
        S16, R16, B16 = 16, 49, 1 << 17
        t16, s16, _ = env.make_synthetic_demos(B16, R16, S16, values, probs, shift, seed=3, device=dev)
        ms = _time_ms(lambda: env.make_synthetic_demos(B16, R16, S16, values, probs, shift, seed=3, device=dev, tape=t16, slab=s16), 3, torch)
        o16, f16, n16 = torch.empty_like(s16), torch.empty(B16, dtype=torch.uint8, device=dev), torch.empty(B16, dtype=torch.int32, device=dev)
        ms_step = _time_ms(lambda: env.step_batch(s16, t16[R16 - 1], S16, shift, out=o16, flags=f16, nnz=n16), 10, torch)
        del o16
        cb16, m16 = basis_block(S16, s16, B16, 0.3)
        ms_cbf = _time_ms(lambda: env.change_of_basis(s16, m16, S16, tape=t16, shift=shift, shift_out=100), 3, torch)
        out["size_16x16x16"] = {"games": B16, "R": R16, "synthetic_demos_per_sec": B16 / ms * 1e3,
                                "demo_hbm_frac": B16 * demo_bytes(S16, R16) / (ms * 1e-3) / 1e9 / peak,
                                "env_steps_per_sec": B16 / ms_step * 1e3, "step_ms": ms_step,
                                "step_hbm_frac": B16 * STEP_BYTES[16] / (ms_step * 1e-3) / 1e9 / peak,
                                "change_of_basis": cb16,
                                "change_of_basis_with_factors_games_per_sec": B16 / ms_cbf * 1e3,
                                "kernel": "basis_mma16_kernel (mma.sync int8 + f16, one warp per game)"}
        del t16, s16, m16
        # BASELINE.json configs[4]: rollout-heavy point, 2^24 games in total x 64 steps fused (the demos' 23 actions, then
        # null actions: a solved game is frozen), action tape resident in HBM
        B5, K5 = (1 << 24) // world, 64
        tape5 = torch.empty((K5, B5, lay.token_pitch), dtype=torch.uint8, device=dev)
        null = torch.zeros(lay.token_pitch, dtype=torch.uint8, device=dev)
        null[: 3 * S] = shift
        tape5[R:] = null
        _, slab5, _ = env.make_synthetic_demos(B5, R, S, values, probs, shift, seed=5, first_demo=rank * B5, device=dev, tape=tape5[:R])
        o5 = torch.empty_like(slab5)
        ms = _time_ms(lambda: env.rollout(slab5, tape5, S, shift, out=o5), 2, torch)
        _, fl5, _, st5 = env.rollout(slab5, tape5, S, shift, out=o5)
        out["config5_rollout_16M_x64"] = {"games_per_gpu": B5, "K": K5, "ms": ms, "nominal_steps_per_sec": B5 * K5 / ms * 1e3,
                                          "applied_steps_per_sec": float(st5.sum().item()) / ms * 1e3,
                                          "solved": int(((fl5 & env.FLAG_TERMINAL) != 0).sum().item()),
                                          "max_steps": int(st5.max().item()), "tape_gib": tape5.numel() / 2 ** 30}
        del tape5, slab5, o5
    if world > 1:
        out["multi_gpu"] = measure_collectives(env, tgd, torch, dev, values, probs, shift, world, rank, barrier)
    return out


def measure_collectives(env, tgd, torch, dev, values, probs, shift, world, rank, barrier) -> dict:
    """N > 1 only: the demo all-gather as its own phase (straight into the full tensor, NVLink-bound, SURVEY 8e) and
    BASELINE.json configs[3]: three size classes in equal game counts, each sharded by game index, generated, gathered
    with NCCL -- and compared byte for byte on every rank with the same demos generated by ONE GPU."""
    import torch.distributed as dist

    res = {}
    S, R = 9, DEMO_R[9]
    lay = env.layout(S)
    n_g = 1 << 18  # demos per rank
    full = torch.empty((n_g * world, lay.game_pitch), dtype=torch.int8, device=dev)
    lo = rank * n_g
    env.make_synthetic_demos(n_g, R, S, values, probs, shift, seed=7, first_demo=lo, device=dev,
                             tape=torch.empty((R, n_g, lay.token_pitch), dtype=torch.uint8, device=dev), slab=full[lo:lo + n_g])
    barrier()
    ms = _time_ms(lambda: tgd.gather_shards(full[lo:lo + n_g], n_g * world, dim=0, out=full), 5, torch)
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    out_bytes = n_g * world * lay.game_pitch
    res["demo_all_gather"] = {"ms": ms, "bytes_out_per_rank": out_bytes, "algbw_gbs": out_bytes / (ms * 1e-3) / 1e9,
                              "busbw_gbs": out_bytes * (world - 1) / world / (ms * 1e-3) / 1e9,
                              "nvlink_frac": out_bytes * (world - 1) / world / (ms * 1e-3) / 1e9 / 900.0,
                              "how": "all_gather_into_tensor in place (the shard is the rank's slice of the output)"}
    del full
    classes = {}
    all_equal = True
    for Sx, vals, prs, sh in ((4, VALUES3, PROBS3, 1), (9, values, probs, shift), (16, values, probs, shift)):
        n_total = (1 << 16) // world * world
        Rx = DEMO_R[Sx]
        tape, slab, flags = tgd.make_synthetic_demos_gathered(n_total, Rx, Sx, vals, prs, sh, seed=11, device=dev)
        t1, s1, f1 = env.make_synthetic_demos(n_total, Rx, Sx, vals, prs, sh, seed=11, first_demo=0, device=dev)
        eq = bool(torch.equal(tape, t1) and torch.equal(slab, s1) and torch.equal(flags, f1))
        e = torch.tensor([1 if eq else 0], device=dev)
        dist.all_reduce(e, op=dist.ReduceOp.MIN)
        classes[f"{Sx}x{Sx}x{Sx}"] = {"demos": n_total, "R": Rx, "bytes": tape.numel() + slab.numel() + flags.numel(),
                                      "gathered_equals_one_gpu_on_every_rank": bool(e.item())}
        all_equal &= bool(e.item())
        del tape, slab, t1, s1
    res["config4_mixed_sizes"] = {"classes": classes, "byte_identical": all_equal, "backend": dist.get_backend(), "ranks": world}
    return res


# ------------------------------------------------------------------------------------------------ main
def main() -> None:
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist

    from mat_mul_b200 import _lib, env
    from mat_mul_b200 import dist as tgd

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_cores = env.bind_host_to_gpu(local)  # pinned staging buffers of the e2e leg land on the GPU's NUMA node
    if world > 1:
        # stdout carries exactly one JSON line: NCCL's own log (its version banner at NCCL_DEBUG=VERSION/WARN, which the GPU
        # boxes export) goes to stderr instead
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # honoured above the VERSION level
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":   # the banner-only level always prints to stdout
            del os.environ["NCCL_DEBUG"]
        dist.init_process_group("nccl", device_id=dev)

    S, shift, B, K, W = args.size, 2, args.games, args.steps, max(args.warmup, 3)
    R = DEMO_R[S]
    lay = env.layout(S)
    if args.ctas_per_sm or args.variant:
        if not _lib.TUNING:
            raise SystemExit("--ctas-per-sm / --variant need the sweep build: TG_TUNING=1")
        _lib.lib().tg_tune_step_ctas_per_sm(args.ctas_per_sm)
        _lib.lib().tg_tune_step_variant(args.variant)

    def barrier() -> None:
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    peak, peak_kind = hbm_peak()
    dump = args.dump_outputs is not None and rank == 0
    if args.metric == "demos":
        blk = measure_demos(env, torch, dist, dev, S, B, R, VALUES5, PROBS5, shift, world, rank, local, barrier, K,
                            not args.no_e2e, not args.no_cpu, dump=dump)
        if dump:
            write_outputs(args.dump_outputs, blk.pop("outputs"))
        if rank == 0:
            line = {"metric": blk["metric"], "value": blk["value"], "unit": blk["unit"], "n_gpus": world, "steps": K, "warmup": 3,
                    "ms_per_step": blk["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                    "dtype": "int8", "data": "synthetic", "config": workload_config("demos", S, B, shift, world),
                    "roofline": blk["roofline"], "e2e": blk.get("e2e"), "gpu_launches": blk["gpu_launches"],
                    "cpu_baseline": blk.get("cpu_baseline"), "cpu_reference": blk.get("cpu_reference"), "clocks": None}
            print(json.dumps(line), flush=True)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    # ---- synthetic games, resident in HBM: the product's own demo generator (Philox stream keyed by the GLOBAL
    # game index, so the union over ranks is independent of N); every game replays its own demo in reverse order
    # (datasets.py:90-92), i.e. a genuine transition on every step; P(coef = 0) = 0.7 as in the reference
    tape3, slab_a, dflags = env.make_synthetic_demos(B, R, S, VALUES5, PROBS5, shift, seed=0x5EED, first_demo=rank * B, device=dev)
    slab0 = slab_a.clone()  # the targets, kept for the full-episode check below
    slab_b = torch.empty_like(slab_a)
    flags = torch.empty(B, dtype=torch.uint8, device=dev)
    nnz = torch.empty(B, dtype=torch.int32, device=dev)

    def one_step(i: int):
        src, dst = (slab_a, slab_b) if i % 2 == 0 else (slab_b, slab_a)
        return env.step_batch(src, tape3[(R - 1 - i) % R], S, shift, out=dst, flags=flags, nnz=nnz)

    for i in range(W):
        one_step(i)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for i in range(K):
        last = one_step(W + i)
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    # copied before the loads below overwrite the buffers
    outputs = sample_outputs({"slab": (last[0], 0), "flags": (last[1], 0), "nnz": (last[2], 0)}, B) if dump else None
    # keep the clock sampler under the same load for ~1 s (its period is 200 ms); results are discarded
    t_end = time.perf_counter() + max(0.0, 1.0 - ms / 1e3)
    i = 0
    scratch_f, scratch_n = torch.empty_like(flags), torch.empty_like(nnz)
    while time.perf_counter() < t_end:
        env.step_batch(slab_a, tape3[i % R], S, shift, out=slab_b, flags=scratch_f, nnz=scratch_n); i += 1
        if i % 8 == 0:
            torch.cuda.synchronize()
    torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    ms = max_over_ranks(ms, torch, dist, dev, world)
    value = world * B * K / (ms / 1e3)

    # ---- full-size correctness property, independent of --steps/--warmup: from the targets, the demos' R actions in reverse
    # bring EVERY game to the zero tensor (per-step launches, the same kernel as the timed region); statistics reduced
    # over ranks with the path's only collective (two tiny all_reduces)
    slab_a.copy_(slab0)
    for i in range(R):
        one_step(i)
    stats = tgd.reduce_episode_stats(flags, nnz)
    slab_a.copy_(slab0)
    del slab0

    # ---- end to end through the C ABI with HOST buffers (tg_step_host): PCIe in + kernel + PCIe out
    e2e = None
    extras_e2e = {}
    if not args.no_e2e:
        Be = B
        h_slab = torch.empty((Be, lay.game_pitch), dtype=torch.int8).pin_memory()
        h_slab.copy_(slab_a[:Be])
        h_tape = torch.empty((Be, lay.token_pitch), dtype=torch.uint8).pin_memory()
        h_tape.copy_(tape3[R - 1][:Be])
        h_out = torch.empty_like(h_slab).pin_memory()
        h_flags = torch.empty(Be, dtype=torch.uint8).pin_memory()
        h_nnz = torch.empty(Be, dtype=torch.int32).pin_memory()
        hs = env.HostStepper(S, local, chunk=1 << 16)
        Ke = max(3, min(K, 10))
        for _ in range(2):
            hs.step(h_slab, h_tape, h_out, h_flags, h_nnz, shift)
        barrier()
        t0 = time.perf_counter()
        for _ in range(Ke):
            hs.step(h_slab, h_tape, h_out, h_flags, h_nnz, shift)  # returns with results in host memory
        dt = max_over_ranks(time.perf_counter() - t0, torch, dist, dev, world)
        h2d, d2h = Be * (lay.game_pitch + lay.token_pitch), Be * (lay.game_pitch + 5)
        barrier()
        ceil_s = max_over_ranks(copy_ceiling(torch, dev, h2d, d2h, Be >> 16, Ke, barrier), torch, dist, dev, world)
        e2e = {"value": world * Be * Ke / dt, "unit": "steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": Ke,
               "api": "tg_step_host (C ABI, pinned host buffers, 64Ki-game chunks through dedicated H2D / kernel / D2H streams chained by events)",
               "host_cores_bound": len(numa_cores),
               "ceiling_gbs": (h2d + d2h) / ceil_s / 1e9, "achieved_gbs": (h2d + d2h) * Ke / dt / 1e9,
               "frac_of_ceiling": ((h2d + d2h) * Ke / dt) / ((h2d + d2h) / ceil_s),
               "ceiling": "the same bytes per step as plain pinned cudaMemcpyAsync in the same chunks, H2D and D2H streams "
                          "concurrently, no kernel, as many repetitions as e2e steps, all ranks at once behind a barrier (max over ranks)"}
        # the K-step host entry (the _take_actions use case, datasets.py:144-153): the slab crosses PCIe once per R steps
        h_tapeK = torch.empty((R, Be, lay.token_pitch), dtype=torch.uint8).pin_memory()
        h_tapeK.copy_(tape3.flip(0))
        h_steps = torch.empty(Be, dtype=torch.int32).pin_memory()
        hs.rollout(h_slab, h_tapeK, h_out, h_flags, h_nnz, h_steps, shift)
        barrier()
        t0 = time.perf_counter()
        for _ in range(3):
            hs.rollout(h_slab, h_tapeK, h_out, h_flags, h_nnz, h_steps, shift)
        dtk = max_over_ranks((time.perf_counter() - t0) / 3, torch, dist, dev, world)
        extras_e2e["rollout_host"] = {"value": world * Be * R / dtk, "unit": "steps/s", "K": R, "games_per_sec": world * Be / dtk,
                                      "solved": int((h_flags & 1).sum().item()), "api": "tg_rollout_host (slab once per K steps)",
                                      "h2d_bytes_per_call": Be * (lay.game_pitch + R * lay.token_pitch),
                                      "d2h_bytes_per_call": Be * (lay.game_pitch + 9)}
        hs.close()
        del h_slab, h_tape, h_out, h_tapeK

    demos = measure_demos(env, torch, dist, dev, S, B, R, VALUES5, PROBS5, shift, world, rank, local, barrier, max(3, min(K, 10)),
                          not args.no_e2e, not args.no_cpu)
    demos4 = None
    if S == 9 and not args.no_extras:
        demos4 = measure_demos(env, torch, dist, dev, 4, 1 << 22, DEMO_R[4], VALUES3, PROBS3, 1, world, rank, local, barrier, 5,
                               False, not args.no_cpu)
    extras = None
    if not args.no_extras:
        extras = measure_extras(env, dev, S, shift, slab_a, tape3, R, VALUES5, PROBS5, world, rank, barrier)
        extras.update(extras_e2e)

    if rank == 0:
        algo = STEP_BYTES[S] * B
        achieved = algo / (ms / K / 1e3) / 1e9
        traffic = None
        tj = ROOT / "profiles" / "traffic.json"
        if tj.exists():
            try:
                traffic = json.loads(tj.read_text()).get(f"step_S{S}_B{B}")
            except Exception:
                traffic = None
        line = {
            "metric": "env_steps_per_sec", "value": value, "unit": "steps/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int8",
            "data": "synthetic", "config": workload_config("steps", S, B, shift, world),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_kind": peak_kind, "kernel": "tg::step_kernel",
                         "algorithmic_bytes_per_step": STEP_BYTES[S],
                         "moved_bytes_per_step": 2 * lay.game_pitch + lay.token_pitch + 5},
            "e2e": e2e, "gpu_launches": K * world, "clocks": clocks,
            "episode_stats": {"games": stats.games, "solved": stats.solved, "min_nnz": stats.min_nnz,
                              "out_of_range": stats.out_of_range,
                              "note": f"from the targets, the demos' {R} actions replayed in reverse by {R} tg_step launches "
                                      "(run after the timed region, independent of --steps/--warmup)",
                              "collective": "all_reduce(SUM), all_reduce(MIN) of 5 int64"},
            "demos": demos, "demos_4x4x4": demos4, "extras": extras,
        }
        if world == 1 and not args.no_cpu:
            v, cores, sample = cpu_step_port(S, shift, 12.0)
            line["cpu_baseline"] = {"value": v, "unit": "steps/s", "cores": cores, "kind": "port", "sample": sample}
            real = cpu_step_reference(S, 5.0)
            if real is not None:
                line["cpu_reference"] = {"value": real[0], "unit": "steps/s", "cores": real[1], "kind": "reference", "sample": real[2]}
        if dump:
            write_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
