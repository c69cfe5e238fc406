"""Batched TensorGame environment on device formats (additions alongside the
reference-named API; the mirrors in utils.py / datasets.py / act.py call these).

All tensors are CUDA tensors owned by PyTorch; kernels run on the current
torch stream through the C ABI (include/tensorgame.h).  Nothing here computes
on the CPU: without the CUDA library or a CUDA tensor these functions raise.
"""
from __future__ import annotations

import ctypes as C
from contextlib import contextmanager
from dataclasses import dataclass

import torch

from . import _lib
from ._lib import (FLAG_EXHAUSTED, FLAG_NULL, FLAG_PATH_EXACT, FLAG_PATH_PLANES, FLAG_RANGE, FLAG_TERMINAL,  # noqa: F401
                   FLAG_TOKEN_RANGE, TensorGameError, check)


@dataclass(frozen=True)
class Layout:
    S: int
    row_pitch: int    # RP: bytes per i-row
    game_pitch: int   # GP: bytes per game in a slab
    token_pitch: int  # TP: bytes per game in a tape

    @property
    def algorithmic_step_bytes(self) -> int:
        """SURVEY.md 8(d): 2*S^3 + 3S + 1 + 4 bytes per env step."""
        return 2 * self.S ** 3 + 3 * self.S + 5


def layout(S: int) -> Layout:
    rp, gp, tp = C.c_int(), C.c_int(), C.c_int()
    check(_lib.lib().tg_layout(S, C.byref(rp), C.byref(gp), C.byref(tp)), f"tg_layout(S={S})")
    return Layout(S, rp.value, gp.value, tp.value)


@contextmanager
def _on(*tensors):
    """Launch context: makes the operands' device current and yields torch's current stream OF THAT DEVICE (so a
    launch lands where the tensors live and is ordered after their producers, whatever the caller's current
    device is).  All operands must share one CUDA device."""
    dev = None
    for t in tensors:
        if t is None:
            continue
        d = t.device
        if d.type != "cuda":
            raise TensorGameError("operands must live on a CUDA device (there is no CPU path)")
        if dev is None:
            dev = d
        elif d != dev:
            raise TensorGameError(f"operands live on different devices ({dev} and {d})")
    with torch.cuda.device(dev):
        yield C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _stream() -> C.c_void_p:
    """torch's current stream on the CURRENT device (for callers that drive the C ABI directly, e.g. the tests)."""
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _call(name: str, operands: tuple, *args) -> None:
    """One C-ABI launch on the operands' device and that device's current torch stream (the stream is the last
    argument of every device entry point of include/tensorgame.h)."""
    with _on(*operands) as st:
        check(getattr(_lib.lib(), name)(*args, st), name)


def _need_cuda(t: torch.Tensor, name: str, dtype: torch.dtype) -> None:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise TensorGameError(f"{name} must be a CUDA tensor (there is no CPU path)")
    if t.dtype != dtype:
        raise TensorGameError(f"{name} must be {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise TensorGameError(f"{name} must be contiguous")


def _p(t: torch.Tensor | None) -> C.c_void_p:
    return C.c_void_p(0 if t is None else t.data_ptr())


_SLAB_SUFFIX = {torch.int16: "_i16", torch.int32: "_gf2"}


def _game_slab(slab: torch.Tensor, name: str = "slab") -> str:
    """Checks a residual slab, int8, int16 (include/tensorgame.h "int16 game path") or an int32 bit slab ("mod-2 game
    path"), and returns the suffix of the entry points for its dtype: "", "_i16" or "_gf2"."""
    sfx = _SLAB_SUFFIX.get(slab.dtype, "") if isinstance(slab, torch.Tensor) else ""
    _need_cuda(slab, name, {"": torch.int8, "_i16": torch.int16, "_gf2": torch.int32}[sfx])
    return sfx


def _game_pitch(sfx: str, S: int) -> int:
    """Elements per game of a slab of the format `sfx` selects."""
    return layout_gf2(S).game_words if sfx == "_gf2" else layout(S).game_pitch


# ---------------------------------------------------------------- formats
def new_slab(B: int, S: int, device) -> torch.Tensor:
    """Zeroed residual slab, int8 (B, GP)."""
    return torch.zeros((B, layout(S).game_pitch), dtype=torch.int8, device=device)


def slab_view(slab: torch.Tensor, S: int) -> torch.Tensor:
    """Strided (B, S, S, S) int8 view of a slab (no copy)."""
    lay = layout(S)
    return slab.as_strided((slab.shape[0], S, S, S), (lay.game_pitch, lay.row_pitch, S, 1))


def pack_states(heads: torch.Tensor, S: int | None = None, out: torch.Tensor | None = None) -> torch.Tensor:
    """float32 heads (B, S, S, S) (any batch stride, dense game) -> slab.  Raises if a value
    is not an integer in [-128, 127]."""
    if heads.dtype != torch.float32 or not heads.is_cuda:
        raise TensorGameError("heads must be a CUDA float32 tensor")
    S = S or heads.shape[-1]
    B = heads.shape[0]
    if heads.shape[1:] != (S, S, S) or heads[0].numel() and not heads[0].is_contiguous():
        raise TensorGameError("heads must be (B, S, S, S) with dense games")
    out = new_slab(B, S, heads.device) if out is None else out
    flag = torch.zeros(1, dtype=torch.int32, device=heads.device)
    stride = heads.stride(0) if B > 1 else S ** 3
    _call("tg_pack_f32", (heads, out, flag,), _p(heads), stride, _p(out), B, S, _p(flag))
    if int(flag.item()):
        raise TensorGameError("pack_states: residual entries must be integers in [-128, 127]")
    return out


def expand_states(slab: torch.Tensor, S: int, out: torch.Tensor | None = None) -> torch.Tensor:
    """slab -> float32 (B, S, S, S) (the dtype model.py consumes).  An int32 bit slab (B, GB/4) gives its 0/1 values
    in one pass (tg_expand_f32_gf2)."""
    bits = isinstance(slab, torch.Tensor) and slab.dtype == torch.int32
    _need_cuda(slab, "slab", torch.int32 if bits else torch.int8)
    if bits and (slab.dim() != 2 or slab.shape[1] != layout_gf2(S).game_words):
        raise TensorGameError(f"expected bits (B,{layout_gf2(S).game_words})")
    B = slab.shape[0]
    if out is None:
        out = torch.empty((B, S, S, S), dtype=torch.float32, device=slab.device)
    stride = out.stride(0) if B > 1 else S ** 3
    _call("tg_expand_f32_gf2" if bits else "tg_expand_f32", (slab, out,), _p(slab), _p(out), stride, B, S)
    return out


def slab16_view(slab16: torch.Tensor, S: int) -> torch.Tensor:
    """Strided (B, S, S, S) int16 view of an int16 slab (no copy)."""
    lay = layout(S)
    return slab16.as_strided((slab16.shape[0], S, S, S), (lay.game_pitch, lay.row_pitch, S, 1))


def pack_states16(heads: torch.Tensor, S: int | None = None) -> torch.Tensor:
    """float32 heads (B, S, S, S) -> int16 slab (B, GP) of int16 (tg_pack_f32_i16): the format for residuals the int8
    slab cannot hold.  Raises if a value is not an integer in [-32768, 32767]."""
    if heads.dtype != torch.float32 or not heads.is_cuda:
        raise TensorGameError("heads must be a CUDA float32 tensor")
    S = S or heads.shape[-1]
    B = heads.shape[0]
    if heads.shape[1:] != (S, S, S) or heads[0].numel() and not heads[0].is_contiguous():
        raise TensorGameError("heads must be (B, S, S, S) with dense games")
    out = torch.empty((B, layout(S).game_pitch), dtype=torch.int16, device=heads.device)
    flag = torch.zeros(1, dtype=torch.int32, device=heads.device)
    stride = heads.stride(0) if B > 1 else S ** 3
    _call("tg_pack_f32_i16", (heads, out, flag), _p(heads), stride, _p(out), B, S, _p(flag))
    if int(flag.item()):
        raise TensorGameError("pack_states16: residual entries must be integers in [-32768, 32767]")
    return out


def expand_states16(slab16: torch.Tensor, S: int, out: torch.Tensor | None = None) -> torch.Tensor:
    """int16 slab -> float32 (B, S, S, S) (tg_expand_f32_i16)."""
    _need_cuda(slab16, "slab16", torch.int16)
    B = slab16.shape[0]
    if out is None:
        out = torch.empty((B, S, S, S), dtype=torch.float32, device=slab16.device)
    stride = out.stride(0) if B > 1 else S ** 3
    _call("tg_expand_f32_i16", (slab16, out), _p(slab16), _p(out), stride, B, S)
    return out


def pack_actions(actions: torch.Tensor, S: int | None = None, rebase: int = 0) -> torch.Tensor:
    """int64 tokens (B, 3S) -> tape uint8 (B, TP).  rebase is added to every token first (a caller whose
    coefficient is token - s passes rebase = 4 - s and then uses shift 4: include/tensorgame.h "Token bound");
    tokens must land in [0, 8], the tape's alphabet."""
    _need_cuda(actions, "actions", torch.int64)
    S = S or actions.shape[-1] // 3
    B = actions.shape[0]
    if rebase:
        actions = actions + rebase
    if B and (int(actions.min()) < 0 or int(actions.max()) > 8):
        raise TensorGameError("pack_actions: factor coefficients must be in [-4, 4] (tape tokens in [0, 8])")
    tape = torch.empty((B, layout(S).token_pitch), dtype=torch.uint8, device=actions.device)
    flag = torch.zeros(1, dtype=torch.int32, device=actions.device)
    _call("tg_pack_actions_i64", (actions, tape, flag,), _p(actions), _p(tape), B, S, _p(flag))
    if int(flag.item()):
        raise TensorGameError("pack_actions: tokens must be in [0, 255]")
    return tape


def unpack_actions(tape: torch.Tensor, S: int) -> torch.Tensor:
    _need_cuda(tape, "tape", torch.uint8)
    B = tape.shape[0]
    out = torch.empty((B, 3 * S), dtype=torch.int64, device=tape.device)
    _call("tg_unpack_actions_i64", (tape, out,), _p(tape), _p(out), B, S)
    return out


# ---------------------------------------------------------------- mod-2 bit slabs
@dataclass(frozen=True)
class LayoutGF2:
    S: int
    row_words: int   # RW: 32-bit words per i-row (S^2 bits)
    game_bytes: int  # GB: bytes per game in a bit slab

    @property
    def game_words(self) -> int:
        return self.game_bytes // 4


def layout_gf2(S: int) -> LayoutGF2:
    rw, gb = C.c_int(), C.c_int()
    check(_lib.lib().tg_layout_gf2(S, C.byref(rw), C.byref(gb)), f"tg_layout_gf2(S={S})")
    return LayoutGF2(S, rw.value, gb.value)


def pack_gf2(slab: torch.Tensor, S: int) -> torch.Tensor:
    """int8 or int16 slab -> bit slab int32 (B, GB/4) of the residues mod 2 (tg_pack_gf2 / tg_pack_gf2_i16: the low bit
    of each two's-complement entry)."""
    sfx = _game_slab(slab)
    if sfx == "_gf2":
        raise TensorGameError("pack_gf2 takes an int8 or int16 slab")
    if slab.dim() != 2 or slab.shape[1] != layout(S).game_pitch:
        raise TensorGameError(f"expected slab (B,{layout(S).game_pitch})")
    B = slab.shape[0]
    bits = torch.empty((B, layout_gf2(S).game_words), dtype=torch.int32, device=slab.device)
    _call("tg_pack_gf2" + sfx, (slab, bits), _p(slab), _p(bits), B, S)
    return bits


def unpack_gf2(bits: torch.Tensor, S: int) -> torch.Tensor:
    """bit slab -> int8 slab of 0/1 values (tg_unpack_gf2); expand_states takes it on to float32."""
    _need_cuda(bits, "bits", torch.int32)
    if bits.dim() != 2 or bits.shape[1] != layout_gf2(S).game_words:
        raise TensorGameError(f"expected bits (B,{layout_gf2(S).game_words})")
    B = bits.shape[0]
    slab = torch.empty((B, layout(S).game_pitch), dtype=torch.int8, device=bits.device)
    _call("tg_unpack_gf2", (bits, slab), _p(bits), _p(slab), B, S)
    return slab


# ---------------------------------------------------------------- K1
def step_batch(slab: torch.Tensor, tape: torch.Tensor, S: int, shift: int, out: torch.Tensor | None = None,
               flags: torch.Tensor | None = None, nnz: torch.Tensor | None = None):
    """One transition for every game: out = slab - u(x)v(x)w.  Returns (out, flags, nnz).

    slab int8, int16 (tg_step_i16) or an int32 bit slab (tg_step_gf2: out = slab xor rank1 mod 2); out has its dtype.  flags uint8 (B,): FLAG_TERMINAL | FLAG_NULL | FLAG_RANGE;
    nnz int32 (B,).  Reference: act.py:266-275, training.py:253-267, utils.py:181-194.
    """
    sfx = _game_slab(slab)
    _need_cuda(tape, "tape", torch.uint8)
    B = slab.shape[0]
    lay, gp = layout(S), _game_pitch(sfx, S)
    if slab.shape != (B, gp) or tape.shape != (B, lay.token_pitch):
        raise TensorGameError(f"expected slab (B,{gp}) and tape (B,{lay.token_pitch})")
    out = torch.empty_like(slab) if out is None else out
    flags = torch.empty(B, dtype=torch.uint8, device=slab.device) if flags is None else flags
    nnz = torch.empty(B, dtype=torch.int32, device=slab.device) if nnz is None else nnz
    _call("tg_step" + sfx, (slab, tape, out, flags, nnz,), _p(slab), _p(tape), _p(out), _p(flags), _p(nnz), B, S, shift)
    return out, flags, nnz


# ---------------------------------------------------------------- K2
def expand_children(slab: torch.Tensor, tape: torch.Tensor, S: int, shift: int, with_keys: bool = True):
    """Batched leaf expansion (tg_expand_children): children[b, c] = slab[b] - rank1(tape[b, c]).

    slab int8 or int16 (B, GP) (tg_expand_children_i16) or a bit slab (tg_expand_children_gf2), tape uint8 (B, k, TP).  Returns (children (B, k, GP) of the
    slab's dtype, flags (B, k), nnz (B, k), keys (B, k) or None).  Reference: act.py:266-275 get_child_states + the
    null / terminal / already-in-tree tests of extend_tree (act.py:177-195), for B states at once."""
    sfx = _game_slab(slab)
    _need_cuda(tape, "tape", torch.uint8)
    lay, gp = layout(S), _game_pitch(sfx, S)
    B = slab.shape[0]
    if tape.dim() != 3 or tape.shape[0] != B or tape.shape[2] != lay.token_pitch or slab.shape[1] != gp:
        raise TensorGameError(f"expected slab (B,{gp}) and tape (B,k,{lay.token_pitch})")
    k = tape.shape[1]
    dev = slab.device
    children = torch.empty((B, k, gp), dtype=slab.dtype, device=dev)
    flags = torch.empty((B, k), dtype=torch.uint8, device=dev)
    nnz = torch.empty((B, k), dtype=torch.int32, device=dev)
    keys = torch.empty((B, k), dtype=torch.int64, device=dev) if with_keys else None
    _call("tg_expand_children" + sfx, (slab, tape, children, flags, nnz, keys,), _p(slab), _p(tape), k, _p(children), _p(flags), _p(nnz), _p(keys), B, S, shift)
    return children, flags, nnz, keys


def rollout(slab: torch.Tensor, tape: torch.Tensor, S: int, shift: int, out: torch.Tensor | None = None):
    """Apply a step-major tape (K, B, TP) to every game, freezing solved games.
    slab int8, int16 (tg_rollout_i16) or a bit slab (tg_rollout_gf2).  Returns (out, flags, nnz, steps).  Reference: datasets.py:144-153,
    training.py:336-342, act.py:49."""
    sfx = _game_slab(slab)
    _need_cuda(tape, "tape", torch.uint8)
    lay, gp = layout(S), _game_pitch(sfx, S)
    B = slab.shape[0]
    if tape.dim() != 3 or tape.shape[1] != B or tape.shape[2] != lay.token_pitch or slab.shape[1] != gp:
        raise TensorGameError(f"expected slab (B,{gp}) and tape (K,B,{lay.token_pitch})")
    K = tape.shape[0]
    out = torch.empty_like(slab) if out is None else out
    flags = torch.empty(B, dtype=torch.uint8, device=slab.device)
    nnz = torch.empty(B, dtype=torch.int32, device=slab.device)
    steps = torch.empty(B, dtype=torch.int32, device=slab.device)
    _call("tg_rollout" + sfx, (slab, tape, out, flags, nnz, steps,), _p(slab), _p(tape), B * lay.token_pitch, K, _p(out), _p(flags), _p(nnz), _p(steps), B, S, shift)
    return out, flags, nnz, steps


def replay(slab: torch.Tensor, tape: torch.Tensor, S: int, shift: int, out: torch.Tensor | None = None):
    """All K actions of a step-major tape applied without freezing (datasets.py:144-153); slab int8, int16
    (tg_replay_i16) or a bit slab (tg_replay_gf2).  Returns (out, flags, nnz)."""
    sfx = _game_slab(slab)
    _need_cuda(tape, "tape", torch.uint8)
    lay, gp = layout(S), _game_pitch(sfx, S)
    B, K = slab.shape[0], tape.shape[0]
    if tape.dim() != 3 or tape.shape[1] != B or tape.shape[2] != lay.token_pitch or slab.shape[1] != gp:
        raise TensorGameError(f"expected slab (B,{gp}) and tape (K,B,{lay.token_pitch})")
    out = torch.empty_like(slab) if out is None else out
    flags = torch.empty(B, dtype=torch.uint8, device=slab.device)
    nnz = torch.empty(B, dtype=torch.int32, device=slab.device)
    _call("tg_replay" + sfx, (slab, tape, out, flags, nnz,), _p(slab), _p(tape), B * lay.token_pitch, K, _p(out), _p(flags), _p(nnz), B, S, shift)
    return out, flags, nnz


# ---------------------------------------------------------------- K3
def _cat_arrays(values, probs):
    import numpy as np

    v = np.ascontiguousarray(values, dtype=np.int8)
    p = np.ascontiguousarray(probs, dtype=np.float64)
    if v.ndim != 1 or v.shape != p.shape or not 1 <= len(v) <= 8:
        raise TensorGameError("values/probs must be 1-D of equal length <= 8")
    return v, p


def make_synthetic_demos(n_demos: int, max_actions: int, S: int, values=(-1, 0, 1), probs=(0.15, 0.7, 0.15),
                         shift: int = 1, seed: int = 0, first_demo: int = 0, device="cuda", max_tries: int = 64,
                         tape: torch.Tensor | None = None, slab: torch.Tensor | None = None):
    """Throughput-mode demo generation (device Philox stream, tg_demo_gen_philox).

    Returns (tape uint8 (R, N, TP) step-major, slab int8 (N, GP), flags uint8 (N,)).
    Same distribution and rejection rule as utils.py:203-233; NOT the torch RNG stream --
    use demos_from_seed for same-seed parity with the reference."""
    lay = layout(S)
    dev = torch.device(device)
    if dev.type != "cuda":
        raise TensorGameError("make_synthetic_demos needs a CUDA device (there is no CPU path)")
    v, p = _cat_arrays(values, probs)
    if tape is None:
        tape = torch.empty((max_actions, n_demos, lay.token_pitch), dtype=torch.uint8, device=dev)
    if slab is None:
        slab = torch.empty((n_demos, lay.game_pitch), dtype=torch.int8, device=dev)
    flags = torch.empty(n_demos, dtype=torch.uint8, device=dev)
    stride = tape.stride(0) if max_actions > 1 else n_demos * lay.token_pitch
    with torch.cuda.device(dev):
        _call("tg_demo_gen_philox", (tape, slab, flags,), seed, first_demo, n_demos, max_actions, S, shift, v.ctypes.data, p.ctypes.data,
                                            len(v), max_tries, _p(tape), stride, _p(slab), _p(flags))
    return tape, slab, flags


def make_synthetic_demos_gf2(n_demos: int, max_actions: int, S: int, values=(-1, 0, 1), probs=(0.15, 0.7, 0.15), shift: int = 1,
                             seed: int = 0, first_demo: int = 0, device="cuda", max_tries: int = 64, tape: torch.Tensor | None = None,
                             bits: torch.Tensor | None = None):
    """Throughput-mode demo generation modulo 2 (tg_demo_gen_gf2): every factor has an odd entry, so no term vanishes mod 2,
    and the targets are bit slabs (the xor of the terms), written without an int8 slab.

    Returns (tape uint8 (R, N, TP) step-major, bits int32 (N, GB/4), flags uint8 (N,): TG_FLAG_EXHAUSTED or 0).  Where 0
    is the only even value of the alphabet, the tape is make_synthetic_demos' for the same arguments and the bits are
    pack_gf2 of its targets."""
    lay, lb = layout(S), layout_gf2(S)
    dev = torch.device(device)
    if dev.type != "cuda":
        raise TensorGameError("make_synthetic_demos_gf2 needs a CUDA device (there is no CPU path)")
    v, p = _cat_arrays(values, probs)
    if tape is None:
        tape = torch.empty((max_actions, n_demos, lay.token_pitch), dtype=torch.uint8, device=dev)
    if bits is None:
        bits = torch.empty((n_demos, lb.game_words), dtype=torch.int32, device=dev)
    flags = torch.empty(n_demos, dtype=torch.uint8, device=dev)
    stride = tape.stride(0) if max_actions > 1 else n_demos * lay.token_pitch
    with torch.cuda.device(dev):
        _call("tg_demo_gen_gf2", (tape, bits, flags), seed, first_demo, n_demos, max_actions, S, shift, v.ctypes.data, p.ctypes.data,
              len(v), max_tries, _p(tape), stride, _p(bits), _p(flags))
    return tape, bits, flags


def accumulate_demos(tape: torch.Tensor, S: int, shift: int, slab: torch.Tensor | None = None):
    """slab[n] = sum_r rank1(tape[r, n]) (tg_demo_accumulate).  Returns (slab, flags)."""
    _need_cuda(tape, "tape", torch.uint8)
    lay = layout(S)
    R, N = tape.shape[0], tape.shape[1]
    if tape.shape[2] != lay.token_pitch:
        raise TensorGameError(f"tape must be (R, N, {lay.token_pitch})")
    if slab is None:
        slab = torch.empty((N, lay.game_pitch), dtype=torch.int8, device=tape.device)
    flags = torch.empty(N, dtype=torch.uint8, device=tape.device)
    _call("tg_demo_accumulate", (tape, slab, flags,), _p(tape), N * lay.token_pitch, N, R, S, shift, _p(slab), _p(flags))
    return slab, flags


def accumulate_demos16(tape: torch.Tensor, S: int, shift: int, slab16: torch.Tensor | None = None):
    """The same sum as accumulate_demos into an int16 slab (tg_demo_accumulate_i16): exact for every tape; the flag
    says an entry does not fit int16.  Where targets beyond the int8 slab's zone go (the reference accumulates them in
    float32 without limit, utils.py:218-232).  Returns (slab16 int16 (N, GP), flags)."""
    _need_cuda(tape, "tape", torch.uint8)
    lay = layout(S)
    R, N = tape.shape[0], tape.shape[1]
    if tape.shape[2] != lay.token_pitch:
        raise TensorGameError(f"tape must be (R, N, {lay.token_pitch})")
    if slab16 is None:
        slab16 = torch.empty((N, lay.game_pitch), dtype=torch.int16, device=tape.device)
    flags = torch.empty(N, dtype=torch.uint8, device=tape.device)
    stride = tape.stride(0) if R > 1 else N * lay.token_pitch
    _call("tg_demo_accumulate_i16", (tape, slab16, flags), _p(tape), stride, N, R, S, shift, _p(slab16), _p(flags))
    return slab16, flags


def torch_cpu_stream(n: int, seed: int | None = None, generator: torch.Generator | None = None, skip: int = 0):
    """The next n doubles torch's CPU generator would produce (torch.rand(dtype=float64)), computed by the
    library's MT19937 (tg_mt19937_fill_f64*) WITHOUT advancing torch's generator.  seed=None continues from
    `generator` (default: the global CPU generator)."""
    import numpy as np

    out = np.empty(n, dtype=np.float64)
    if seed is not None:
        check(_lib.lib().tg_mt19937_fill_f64(seed & 0xFFFFFFFF, skip, n, out.ctypes.data), "tg_mt19937_fill_f64")
        return out
    st = (generator.get_state() if generator is not None else torch.get_rng_state()).numpy().tobytes()
    # at::mt19937 state blob: seed u64 | left i32 | seeded i32 | next u64 | state[624] u64 ...; `left` numbers remain
    # before the next twist, so the read position is 624 - left + 1 (a freshly seeded generator has left == 1)
    pos = 624 - int.from_bytes(st[8:12], "little", signed=True) + 1
    words = np.frombuffer(st, dtype=np.uint64, count=624, offset=24).astype(np.uint32)
    check(_lib.lib().tg_mt19937_fill_f64_state(words.ctypes.data, pos, skip, n, out.ctypes.data), "tg_mt19937_fill_f64_state")
    return out


def demos_from_ustream(ustream, n_demos: int, max_actions: int, S: int, values, probs, shift: int, device="cuda"):
    """Parity-mode demos from an explicit uniform stream (numpy float64, host).  Returns
    (tape (R,N,TP), slab (N,GP), flags (N,), demos_done, doubles_consumed)."""
    import numpy as np

    lay = layout(S)
    dev = torch.device(device)
    if dev.type != "cuda":
        raise TensorGameError("demos_from_ustream needs a CUDA device (there is no CPU path)")
    v = np.ascontiguousarray(values, dtype=np.int8)
    p = np.ascontiguousarray(probs, dtype=np.float32)
    u = torch.from_numpy(np.ascontiguousarray(ustream, dtype=np.float64)).to(dev)
    n_u = u.numel()
    tape = torch.zeros((max_actions, n_demos, lay.token_pitch), dtype=torch.uint8, device=dev)
    slab = torch.empty((n_demos, lay.game_pitch), dtype=torch.int8, device=dev)
    flags = torch.empty(n_demos, dtype=torch.uint8, device=dev)
    result = torch.zeros(2, dtype=torch.int64, device=dev)
    ws_bytes = int(_lib.lib().tg_demo_from_ustream_workspace(n_u, S))
    ws = torch.empty(ws_bytes + 16, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _call("tg_demo_from_ustream", (u, tape, slab, flags, result, ws,), _p(u), n_u, v.ctypes.data, p.ctypes.data, len(v), max_actions, S, shift, n_demos,
                                              _p(tape), n_demos * lay.token_pitch, _p(slab), _p(flags), _p(result), _p(ws),
                                              ws_bytes)
    done, consumed = (int(x) for x in result.tolist())
    return tape, slab, flags, done, consumed


def demos_from_seed(n_demos: int, max_actions: int, S: int, values=(-1, 0, 1), probs=(0.15, 0.7, 0.15), shift: int = 1,
                    seed: int | None = None, generator: torch.Generator | None = None, device="cuda", advance: bool = True):
    """Same demos as the reference's loop (utils.py:203-233 / datasets.py:124-142) run from torch's CPU
    generator: seed=None continues from the global (or given) generator and, if advance, leaves it where
    the reference would have left it.  Returns (tape, slab, flags, doubles_consumed)."""
    import numpy as np

    pv = np.asarray(probs, dtype=np.float64)
    p0 = float(pv[np.asarray(values) == 0].sum() / pv.sum())
    accept = max((1.0 - p0 ** S) ** 3, 1e-3)
    n_u = int(n_demos * max_actions * 3 * S / accept * 1.25) + 64 * 3 * S
    while True:
        u = torch_cpu_stream(n_u, seed=seed, generator=generator)
        tape, slab, flags, done, consumed = demos_from_ustream(u, n_demos, max_actions, S, values, probs, shift, device)
        if done == n_demos:
            break
        n_u *= 2
    if seed is None and advance:  # move torch's generator to where the reference loop would have left it
        left = consumed
        while left > 0:
            k = min(left, 1 << 22)
            torch.rand(k, dtype=torch.float64, generator=generator)
            left -= k
    return tape, slab, flags, consumed


def accumulate_demos_tc(tape: torch.Tensor, shift: int, slab: torch.Tensor | None = None):
    """accumulate_demos for S = 16, R <= 64 on the tensor cores (tg_demo_accumulate_tc, experimental: tcgen05.mma
    kind::i8, accumulators in TMEM).  Entries beyond int8 are stored saturated.  Returns (slab, flags)."""
    _need_cuda(tape, "tape", torch.uint8)
    lay = layout(16)
    R, N = tape.shape[0], tape.shape[1]
    if tape.shape[2] != lay.token_pitch:
        raise TensorGameError(f"tape must be (R, N, {lay.token_pitch})")
    if slab is None:
        slab = torch.empty((N, lay.game_pitch), dtype=torch.int8, device=tape.device)
    flags = torch.empty(N, dtype=torch.uint8, device=tape.device)
    _call("tg_demo_accumulate_tc", (tape, slab, flags,), _p(tape), N * lay.token_pitch, N, R, 16, shift, _p(slab), _p(flags))
    return slab, flags


# ---------------------------------------------------------------- K4 / K6 / K7
def demo_samples(tape: torch.Tensor, slab: torch.Tensor, idx: torch.Tensor, S: int, dim_t: int, replay_shift: int = 1):
    """Batch of SyntheticDemoDataset.__getitem__ results (datasets.py:77-122) from the in-HBM demo store.
    Returns (states f32 (nb,dim_t,S,S,S), scalars f32 (nb,1), actions i64 (nb,3S), rewards f32 (nb,1))."""
    _need_cuda(tape, "tape", torch.uint8)
    _need_cuda(slab, "slab", torch.int8)
    _need_cuda(idx, "idx", torch.int64)
    lay = layout(S)
    R, N = tape.shape[0], tape.shape[1]
    nb = idx.numel()
    dev = tape.device
    states = torch.empty((nb, dim_t, S, S, S), dtype=torch.float32, device=dev)
    scalars = torch.empty((nb, 1), dtype=torch.float32, device=dev)
    actions = torch.empty((nb, 3 * S), dtype=torch.int64, device=dev)
    rewards = torch.empty((nb, 1), dtype=torch.float32, device=dev)
    _call("tg_demo_sample", (tape, slab, idx, states, scalars, actions, rewards,), _p(tape), N * lay.token_pitch, _p(slab), N, R, S, dim_t, replay_shift, _p(idx), nb,
                                    _p(states), _p(scalars), _p(actions), _p(rewards))
    return states, scalars, actions, rewards


class DemoStore:
    """The in-HBM demonstration store the training-sample batcher reads (replaces the two .pt files per demo of
    datasets.py:62-69): demo-major action records uint8 (N, R, TP) -- the records a .. R-1 one sample needs are one
    contiguous run -- and the targets as an int8 slab, or an int16 slab when a target left the int8 zone.

    Modulo 2 the targets are an int32 bit slab (N, GB/4): samples() then returns the states mod 2 as 0/1 floats
    (tg_demo_sample_gf2) and target_bound is ignored.  Generated demos for a mod-2 run come from
    make_synthetic_demos_gf2, which writes the bit targets directly and conditions every factor on an odd entry (no term
    vanishes mod 2).  For any other tape, replay(zeros, tape, S, shift) of a zeroed bit slab xors the demo's terms into
    it, and pack_gf2 of make_synthetic_demos' int8 targets gives the same bits (RANGE-flagged ones included: they keep
    their parity)."""

    def __init__(self, records: torch.Tensor, targets: torch.Tensor, S: int, shift: int, target_bound: int | None = None):
        _need_cuda(records, "records", torch.uint8)
        lay = layout(S)
        if records.dim() != 3 or records.shape[2] != lay.token_pitch:
            raise TensorGameError(f"records must be (N, R, {lay.token_pitch})")
        self.bits = targets.dtype == torch.int32
        pitch = layout_gf2(S).game_words if self.bits else lay.game_pitch
        if targets.dtype not in (torch.int8, torch.int16, torch.int32) or targets.shape != (records.shape[0], pitch) or not targets.is_cuda:
            raise TensorGameError(f"targets must be an int8 or int16 slab (N, {lay.game_pitch}) or an int32 bit slab "
                                  f"(N, {layout_gf2(S).game_words})")
        self.records, self.targets, self.S, self.shift = records, targets.contiguous(), S, shift
        self.N, self.R = records.shape[0], records.shape[1]
        if self.bits:
            target_bound = 0
        elif target_bound is None:
            target_bound = 127 if targets.dtype == torch.int8 else (int(targets.abs().max()) if self.N else 0)
        self.target_bound = int(target_bound)

    @classmethod
    def from_tape(cls, tape: torch.Tensor, targets: torch.Tensor, S: int, shift: int) -> "DemoStore":
        """From a step-major tape (R, N, TP) (tg_tape_to_demo_major) and its target slab."""
        _need_cuda(tape, "tape", torch.uint8)
        R, N = tape.shape[0], tape.shape[1]
        records = torch.empty((N, R, tape.shape[2]), dtype=torch.uint8, device=tape.device)
        stride = tape.stride(0) if R > 1 else N * tape.shape[2]
        _call("tg_tape_to_demo_major", (tape, records), _p(tape), stride, _p(records), N, R, S)
        return cls(records, targets, S, shift)

    def tape(self) -> torch.Tensor:
        """The step-major view (R, N, TP) of the records (a strided view, no copy)."""
        return self.records.transpose(0, 1)

    def samples(self, idx: torch.Tensor, dim_t: int, replay_shift: int = 1):
        """Batch of SyntheticDemoDataset.__getitem__ results (datasets.py:77-122) for sample indices demo * R + action
        (tg_demo_sample_dm; with bit targets tg_demo_sample_gf2, states mod 2 as 0/1).  Returns (states f32
        (nb,dim_t,S,S,S), scalars f32 (nb,1), actions i64 (nb,3S), rewards f32 (nb,1))."""
        _need_cuda(idx, "idx", torch.int64)
        S, nb, dev = self.S, idx.numel(), self.records.device
        states = torch.empty((nb, dim_t, S, S, S), dtype=torch.float32, device=dev)
        scalars = torch.empty((nb, 1), dtype=torch.float32, device=dev)
        actions = torch.empty((nb, 3 * S), dtype=torch.int64, device=dev)
        rewards = torch.empty((nb, 1), dtype=torch.float32, device=dev)
        operands = (self.records, self.targets, idx, states, scalars, actions, rewards)
        outputs = (_p(idx), nb, _p(states), _p(scalars), _p(actions), _p(rewards))
        if self.bits:
            _call("tg_demo_sample_gf2", operands, _p(self.records), _p(self.targets), self.N, self.R, S, dim_t, replay_shift, *outputs)
        else:
            _call("tg_demo_sample_dm", operands, _p(self.records), _p(self.targets), int(self.targets.dtype == torch.int16),
                  self.target_bound, self.N, self.R, S, dim_t, replay_shift, *outputs)
        return states, scalars, actions, rewards


def slice_rank(slab: torch.Tensor, S: int) -> torch.Tensor:
    """get_rank per game (utils.py:134-140) of an int8 or int16 slab (tg_slice_rank_i16): int32 (B,).  Of a bit slab
    (tg_slice_rank_gf2): the sum of the slices' ranks over GF(2)."""
    sfx = _game_slab(slab)
    ranks = torch.empty(slab.shape[0], dtype=torch.int32, device=slab.device)
    _call("tg_slice_rank" + sfx, (slab, ranks,), _p(slab), _p(ranks), slab.shape[0], S)
    return ranks


def episode_returns(final_slab: torch.Tensor, steps: torch.Tensor, S: int, max_len: int | None = None):
    """The played-game return rule of actor_prediction (act.py:59-62) for a batch of finished games:
    reward_seq = cumsum([-1] * (n - 1) + [-1 - get_rank(final state)]) with n = steps[b] actions played, i.e.
    -1, -2, ..., -(n-1), -n - rank; the rank is tg_slice_rank of the final head (0 for a solved game).
    Returns (returns int64 (B,) = reward_seq[n-1], reward_seq int64 (B, K) zero-padded beyond n, ranks int32 (B,))."""
    ranks = slice_rank(final_slab, S)
    n = steps.to(torch.int64)
    r = ranks.to(torch.int64)
    K = int(max_len if max_len is not None else (int(n.max()) if n.numel() else 0))
    t = torch.arange(1, K + 1, device=n.device, dtype=torch.int64).unsqueeze(0)
    seq = torch.where(t == n.unsqueeze(1), -t - r.unsqueeze(1), -t)
    seq = torch.where(t <= n.unsqueeze(1), seq, torch.zeros_like(seq))
    return -n - r, seq, ranks


def state_keys(slab: torch.Tensor, S: int) -> torch.Tensor:
    """64-bit state keys (as int64 bit patterns), replacing utils.state_to_str dict keys.  An int16 slab
    (tg_state_key_i16) gives the same key as an int8 slab of the same values, a bit slab (tg_state_key_gf2) the key of
    its 0/1 values."""
    sfx = _game_slab(slab)
    keys = torch.empty(slab.shape[0], dtype=torch.int64, device=slab.device)
    _call("tg_state_key" + sfx, (slab, keys,), _p(slab), _p(keys), slab.shape[0], S)
    return keys


# ---------------------------------------------------------------- K5
def sample_unimodular(n: int, S: int, seed: int = 0, first: int = 0, p_nonzero: float = 0.3, device="cuda") -> torch.Tensor:
    """Random unimodular (A, B, C) per game: int8 (n, 3, S, S) (tg_sample_unimodular)."""
    dev = torch.device(device)
    if dev.type != "cuda":
        raise TensorGameError("sample_unimodular needs a CUDA device (there is no CPU path)")
    mats = torch.empty((n, 3, S, S), dtype=torch.int8, device=dev)
    with torch.cuda.device(dev):
        _call("tg_sample_unimodular", (mats,), seed, first, n, S, float(p_nonzero), _p(mats))
    return mats


def change_of_basis(slab: torch.Tensor, mats: torch.Tensor, S: int, tape: torch.Tensor | None = None, shift: int = 0,
                    shift_out: int | None = None, out: torch.Tensor | None = None, out_dtype: torch.dtype = torch.int8,
                    return_path_stats: bool = False):
    """T' = T x1 A x2 B x3 C (and u' = A u, v' = B v, w' = C w for a step-major tape).

    mats int8 (N, 3, S, S) per game or (1, 3, S, S) / (3, S, S) shared.  The result is an int8 slab (flag RANGE: an
    entry left [-64, 63]) or, with out_dtype / out of torch.int16, an int16 slab (SURVEY 8(d)'s format; flag RANGE: an
    entry does not fit int16).  Returns (slab', flags) or (slab', tape', flags); with return_path_stats a dict counting
    the games per kernel path is appended.  Not in the reference: AlphaTensor paper, Methods "Change of basis"."""
    _need_cuda(slab, "slab", torch.int8)
    _need_cuda(mats, "mats", torch.int8)
    N = slab.shape[0]
    m = mats.reshape(-1, 3, S, S)
    if m.shape[0] not in (1, N):
        raise TensorGameError("mats must hold one (A,B,C) triple or one per game")
    per_game = int(m.shape[0] == N and N > 1)
    if out is None:
        out = torch.empty(slab.shape, dtype=out_dtype, device=slab.device)
    if out.dtype not in (torch.int8, torch.int16) or out.shape != slab.shape or not out.is_contiguous():
        raise TensorGameError("out must be a contiguous int8 or int16 slab of the input's shape")
    flags = torch.zeros(N, dtype=torch.uint8, device=slab.device)
    name = "tg_change_of_basis_i16" if out.dtype == torch.int16 else "tg_change_of_basis"
    _call(name, (slab, m, out, flags), _p(slab), _p(m), per_game, _p(out), _p(flags), N, S)
    stats = None
    if return_path_stats:
        exact = int(((flags & FLAG_PATH_EXACT) != 0).sum().item())
        planes = int(((flags & FLAG_PATH_PLANES) != 0).sum().item())
        stats = {"games": N, "fast_path": N - exact - planes, "byte_plane_path": planes, "exact_int32_redo": exact}
    if tape is None:
        return (out, flags, stats) if return_path_stats else (out, flags)
    _need_cuda(tape, "tape", torch.uint8)
    lay = layout(S)
    R = tape.shape[0]
    shift_out = shift if shift_out is None else shift_out
    tape_out = torch.empty_like(tape)
    _call("tg_change_of_basis_factors", (tape, m, tape_out, flags), _p(tape), N * lay.token_pitch, shift, _p(m), per_game,
          _p(tape_out), N * lay.token_pitch, shift_out, _p(flags), N, R, S)
    return (out, tape_out, flags, stats) if return_path_stats else (out, tape_out, flags)


# ---------------------------------------------------------------- K5 mod 2
def sample_invertible_gf2(n: int, S: int, seed: int = 0, first: int = 0, p_nonzero: float = 0.3, device="cuda") -> torch.Tensor:
    """Random (A, B, C) per game, each invertible over GF(2), as bit matrices int32 (n, 3, S): word r of a matrix is its
    row r, bit c its entry (r, c) (tg_sample_invertible_gf2).  At S <= 16 these are sample_unimodular(n, S, seed, first,
    p_nonzero) mod 2."""
    dev = torch.device(device)
    if dev.type != "cuda":
        raise TensorGameError("sample_invertible_gf2 needs a CUDA device (there is no CPU path)")
    mats = torch.empty((n, 3, S), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _call("tg_sample_invertible_gf2", (mats,), seed, first, n, S, float(p_nonzero), _p(mats))
    return mats


def change_of_basis_gf2(bits: torch.Tensor, mats: torch.Tensor, S: int, tape: torch.Tensor | None = None, shift: int = 1,
                        shift_out: int | None = None, out: torch.Tensor | None = None):
    """T' = T x1 A x2 B x3 C over GF(2) on a bit slab (tg_change_of_basis_gf2), and u' = A u, v' = B v, w' = C w mod 2
    for a step-major tape (R, N, TP) (tg_change_of_basis_factors_gf2: tokens read with `shift`, written as residue +
    shift_out, default shift).  mats: bit matrices int32 (N, 3, S) per game, or (1, 3, S) / (3, S) shared.  out may be
    bits (in place).  Returns bits', or (bits', tape') when a tape is given.  Nothing can leave the format mod 2, so there
    are no flags.  Not in the reference: AlphaTensor paper, Methods "Change of basis", in modular arithmetic."""
    _need_cuda(bits, "bits", torch.int32)
    _need_cuda(mats, "mats", torch.int32)
    gw = layout_gf2(S).game_words
    N = bits.shape[0]
    if bits.shape != (N, gw):
        raise TensorGameError(f"expected bits (N,{gw})")
    m = mats.reshape(-1, 3, S)
    if m.shape[0] not in (1, N):
        raise TensorGameError("mats must hold one (A,B,C) triple or one per game")
    per_game = int(m.shape[0] == N and N > 1)
    out = torch.empty_like(bits) if out is None else out
    _need_cuda(out, "out", torch.int32)
    if out.shape != bits.shape:
        raise TensorGameError("out must be a bit slab of the input's shape")
    _call("tg_change_of_basis_gf2", (bits, m, out), _p(bits), _p(m), per_game, _p(out), N, S)
    if tape is None:
        return out
    _need_cuda(tape, "tape", torch.uint8)
    tp = layout(S).token_pitch
    if tape.dim() != 3 or tape.shape[1:] != (N, tp):
        raise TensorGameError(f"tape must be (R, N, {tp})")
    tape_out = torch.empty_like(tape)
    if tape.shape[0] == 0:
        return out, tape_out
    _call("tg_change_of_basis_factors_gf2", (tape, m, tape_out), _p(tape), N * tp, shift, _p(m), per_game, _p(tape_out), N * tp,
          shift if shift_out is None else shift_out, N, tape.shape[0], S)
    return out, tape_out


def bind_host_to_gpu(device: int = 0) -> list[int]:
    """Pin the calling process to the CPU cores that are local to GPU `device` (NVML cpu affinity), so that the
    pinned host buffers it allocates next are first-touched on that GPU's NUMA node.  Matters for the host-buffer
    entry points (tg_step_host) when several ranks share one box.  Returns the cores (empty if unavailable)."""
    import os

    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(device)
        n_words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n_words)
        cores = [64 * w + b for w, word in enumerate(mask) for b in range(64) if (int(word) >> b) & 1]
        allowed = sorted(set(cores) & set(os.sched_getaffinity(0)))
        if allowed:
            os.sched_setaffinity(0, allowed)
        return allowed
    except Exception:
        return []


class HostStepper:
    """End-to-end step for callers whose data lives in host memory (pinned
    numpy/torch CPU buffers): chunked H2D -> tg_step -> D2H over three streams
    inside the C library (tg_step_host)."""

    def __init__(self, S: int, device: int = 0, chunk: int = 1 << 16):
        self.S, self.lay = S, layout(S)
        self._ctx = C.c_void_p()
        check(_lib.lib().tg_host_ctx_create(C.byref(self._ctx), device, S, chunk), "tg_host_ctx_create")

    def step(self, slab: torch.Tensor, tape: torch.Tensor, out: torch.Tensor, flags: torch.Tensor, nnz: torch.Tensor,
             shift: int) -> None:
        for t in (slab, tape, out, flags, nnz):
            if t.is_cuda or not t.is_contiguous():
                raise TensorGameError("HostStepper takes contiguous CPU tensors")
        B = slab.shape[0]
        check(_lib.lib().tg_step_host(self._ctx, _p(slab), _p(tape), _p(out), _p(flags), _p(nnz), B, shift), "tg_step_host")

    def rollout(self, slab: torch.Tensor, tape: torch.Tensor, out: torch.Tensor, flags: torch.Tensor, nnz: torch.Tensor,
                steps: torch.Tensor, shift: int) -> None:
        """K fused steps per PCIe round trip (tg_rollout_host): tape is the dense step-major CPU tape (K, B, TP)."""
        for t in (slab, tape, out, flags, nnz, steps):
            if t.is_cuda or not t.is_contiguous():
                raise TensorGameError("HostStepper takes contiguous CPU tensors")
        K, B = tape.shape[0], slab.shape[0]
        check(_lib.lib().tg_rollout_host(self._ctx, _p(slab), _p(tape), K, _p(out), _p(flags), _p(nnz), _p(steps), B, shift),
              "tg_rollout_host")

    def make_demos(self, tape: torch.Tensor, slab: torch.Tensor, flags: torch.Tensor, shift: int, values, probs, seed: int = 0,
                   first_demo: int = 0, max_tries: int = 64) -> None:
        """Synthetic demonstrations straight into CPU buffers (tg_demo_gen_host): tape (R, N, TP), slab (N, GP), flags (N,)."""
        for t in (tape, slab, flags):
            if t.is_cuda or not t.is_contiguous():
                raise TensorGameError("HostStepper takes contiguous CPU tensors")
        v, p = _cat_arrays(values, probs)
        R, N = tape.shape[0], tape.shape[1]
        check(_lib.lib().tg_demo_gen_host(self._ctx, seed, first_demo, N, R, shift, v.ctypes.data, p.ctypes.data, len(v), max_tries,
                                          _p(tape), _p(slab), _p(flags)), "tg_demo_gen_host")

    def close(self) -> None:
        if self._ctx:
            _lib.lib().tg_host_ctx_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
