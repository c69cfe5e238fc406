"""Batched TensorGame environment on device formats (additions alongside the
reference-named API; the mirrors in utils.py / datasets.py / act.py call these).

All tensors are CUDA tensors owned by PyTorch; kernels run on the current
torch stream through the C ABI (include/tensorgame.h).  Nothing here computes
on the CPU: without the CUDA library or a CUDA tensor these functions raise.
"""
from __future__ import annotations

import ctypes as C
import functools
import math
from contextlib import contextmanager
from dataclasses import dataclass

import torch

from . import _lib
from ._lib import (FLAG_EXHAUSTED, FLAG_NULL, FLAG_PATH_EXACT, FLAG_PATH_PLANES, FLAG_RANGE, FLAG_SINGULAR,  # noqa: F401
                   FLAG_TERMINAL, FLAG_TOKEN_RANGE, TensorGameError, check)


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


@functools.lru_cache(maxsize=None)
def layout(S: int) -> Layout:
    rp, gp, tp = C.c_int(), C.c_int(), C.c_int()
    check(_lib.lib().tg_layout(S, C.byref(rp), C.byref(gp), C.byref(tp)), f"tg_layout(S={S})")
    return Layout(S, rp.value, gp.value, tp.value)


def _device(*tensors) -> torch.device:
    """The one CUDA device every operand lives on."""
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
    return dev


@contextmanager
def _on(*tensors):
    """Launch context: makes the operands' device current and yields torch's current stream OF THAT DEVICE (so a
    launch lands where the tensors live and is ordered after their producers, whatever the caller's current
    device is).  All operands must share one CUDA device."""
    dev = _device(*tensors)
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


def _operand(t: torch.Tensor, name: str, dtype: torch.dtype, shape: tuple | None = None, rows: bool = False) -> torch.Tensor:
    """Checks a tensor before it is handed to the library, whose kernels trust every extent: its dtype, its exact shape
    (a str stands for an extent the call takes from the tensor; None takes any shape) and its layout, contiguous or,
    with rows, dense in every dimension but the first (games of a batch at any stride, or the steps of a step-major
    tape that is a view into a larger store).  The device is checked at launch (_on), after every operand's shape."""
    if not isinstance(t, torch.Tensor):
        raise TensorGameError(f"{name} must be a tensor")
    if t.dtype != dtype or shape is not None and t.shape != shape and (
            t.dim() != len(shape) or any(not isinstance(w, str) and w != n for w, n in zip(shape, t.shape))):
        want = "" if shape is None else f" ({', '.join(map(str, shape))})"
        raise TensorGameError(f"{name} must be {str(dtype)[6:]}{want}, got {str(t.dtype)[6:]} {tuple(t.shape)}")
    if rows:
        step = 1
        for n, s in zip(reversed(t.shape[1:]), reversed(t.stride()[1:])):
            if n != 1 and s != step:
                raise TensorGameError(f"{name} must be dense in every dimension but the first")
            step *= n
    elif not t.is_contiguous():
        raise TensorGameError(f"{name} must be contiguous")
    return t


def _p(t: torch.Tensor | None) -> C.c_void_p:
    return C.c_void_p(0 if t is None else t.data_ptr())


_SLAB_SUFFIX = {torch.int8: "", torch.int16: "_i16", torch.int32: "_gf2"}
_SLAB_DTYPE = {sfx: dtype for dtype, sfx in _SLAB_SUFFIX.items()}


def _game_pitch(sfx: str, S: int) -> int:
    """Elements per game of a slab of the format `sfx` selects."""
    return layout_gf2(S).game_words if sfx == "_gf2" else layout(S).game_pitch


def _slab(t: torch.Tensor, name: str, S: int, sfx: str, B: int | str = "B") -> torch.Tensor:
    """Checks a slab of the format `sfx` selects: int8 or int16 (B, GP), or an int32 bit slab (B, GB/4)."""
    return _operand(t, name, _SLAB_DTYPE[sfx], (B, _game_pitch(sfx, S)))


def _game_slab(slab: torch.Tensor, S: int, name: str = "slab", B: int | str = "B") -> str:
    """Checks a residual slab, int8, int16 (include/tensorgame.h "int16 game path") or an int32 bit slab ("mod-2 game
    path"), and returns the suffix of the entry points for its dtype: "", "_i16" or "_gf2"."""
    sfx = _SLAB_SUFFIX.get(getattr(slab, "dtype", None), "")
    _slab(slab, name, S, sfx, B)
    return sfx


# ---------------------------------------------------------------- formats
def new_slab(B: int, S: int, device) -> torch.Tensor:
    """Zeroed residual slab, int8 (B, GP)."""
    return torch.zeros((B, layout(S).game_pitch), dtype=torch.int8, device=device)


def slab_view(slab: torch.Tensor, S: int) -> torch.Tensor:
    """Strided (B, S, S, S) int8 view of a slab (no copy)."""
    lay = layout(S)
    return slab.as_strided((slab.shape[0], S, S, S), (lay.game_pitch, lay.row_pitch, S, 1))


def _pack(heads: torch.Tensor, S: int | None, out: torch.Tensor | None, sfx: str) -> torch.Tensor:
    """pack_states ("") and pack_states16 ("_i16")."""
    S = S or heads.shape[-1]
    _operand(heads, "heads", torch.float32, ("B", S, S, S), rows=True)
    B = heads.shape[0]
    if out is None:
        out = torch.empty((B, layout(S).game_pitch), dtype=_SLAB_DTYPE[sfx], device=heads.device)
    _slab(out, "out", S, sfx, B)
    flag = torch.zeros(1, dtype=torch.int32, device=heads.device)
    stride = heads.stride(0) if B > 1 else S ** 3
    _call("tg_pack_f32" + sfx, (heads, out, flag), _p(heads), stride, _p(out), B, S, _p(flag))
    if int(flag.item()):
        name, bound = ("pack_states16", "[-32768, 32767]") if sfx else ("pack_states", "[-128, 127]")
        raise TensorGameError(f"{name}: residual entries must be integers in {bound}")
    return out


def _expand(slab: torch.Tensor, name: str, S: int, out: torch.Tensor | None, sfx: str) -> torch.Tensor:
    """expand_states ("" or "_gf2") and expand_states16 ("_i16")."""
    B = _slab(slab, name, S, sfx).shape[0]
    if out is None:
        out = torch.empty((B, S, S, S), dtype=torch.float32, device=slab.device)
    _operand(out, "out", torch.float32, (B, S, S, S), rows=True)
    stride = out.stride(0) if B > 1 else S ** 3
    _call("tg_expand_f32" + sfx, (slab, out), _p(slab), _p(out), stride, B, S)
    return out


def pack_states(heads: torch.Tensor, S: int | None = None, out: torch.Tensor | None = None) -> torch.Tensor:
    """float32 heads (B, S, S, S) (any batch stride, dense game) -> slab.  Raises if a value
    is not an integer in [-128, 127]."""
    return _pack(heads, S, out, "")


def expand_states(slab: torch.Tensor, S: int, out: torch.Tensor | None = None) -> torch.Tensor:
    """slab -> float32 (B, S, S, S) (the dtype model.py consumes; out may have any batch stride).  An int32 bit slab
    (B, GB/4) gives its 0/1 values in one pass (tg_expand_f32_gf2)."""
    return _expand(slab, "slab", S, out, "_gf2" if getattr(slab, "dtype", None) == torch.int32 else "")


def slab16_view(slab16: torch.Tensor, S: int) -> torch.Tensor:
    """Strided (B, S, S, S) int16 view of an int16 slab (no copy)."""
    lay = layout(S)
    return slab16.as_strided((slab16.shape[0], S, S, S), (lay.game_pitch, lay.row_pitch, S, 1))


def pack_states16(heads: torch.Tensor, S: int | None = None) -> torch.Tensor:
    """float32 heads (B, S, S, S) -> int16 slab (B, GP) of int16 (tg_pack_f32_i16): the format for residuals the int8
    slab cannot hold.  Raises if a value is not an integer in [-32768, 32767]."""
    return _pack(heads, S, None, "_i16")


def expand_states16(slab16: torch.Tensor, S: int, out: torch.Tensor | None = None) -> torch.Tensor:
    """int16 slab -> float32 (B, S, S, S) (tg_expand_f32_i16)."""
    return _expand(slab16, "slab16", S, out, "_i16")


def pack_actions(actions: torch.Tensor, S: int | None = None, rebase: int = 0) -> torch.Tensor:
    """int64 tokens (B, 3S) -> tape uint8 (B, TP).  rebase is added to every token first (a caller whose
    coefficient is token - s passes rebase = 4 - s and then uses shift 4: include/tensorgame.h "Token bound");
    tokens must land in [0, 8], the tape's alphabet."""
    S = S or actions.shape[-1] // 3
    B = _operand(actions, "actions", torch.int64, ("B", 3 * S)).shape[0]
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
    B = _operand(tape, "tape", torch.uint8, ("B", layout(S).token_pitch)).shape[0]
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


@functools.lru_cache(maxsize=None)
def layout_gf2(S: int) -> LayoutGF2:
    rw, gb = C.c_int(), C.c_int()
    check(_lib.lib().tg_layout_gf2(S, C.byref(rw), C.byref(gb)), f"tg_layout_gf2(S={S})")
    return LayoutGF2(S, rw.value, gb.value)


def pack_gf2(slab: torch.Tensor, S: int) -> torch.Tensor:
    """int8 or int16 slab -> bit slab int32 (B, GB/4) of the residues mod 2 (tg_pack_gf2 / tg_pack_gf2_i16: the low bit
    of each two's-complement entry)."""
    sfx = _game_slab(slab, S)
    if sfx == "_gf2":
        raise TensorGameError("pack_gf2 takes an int8 or int16 slab")
    B = slab.shape[0]
    bits = torch.empty((B, layout_gf2(S).game_words), dtype=torch.int32, device=slab.device)
    _call("tg_pack_gf2" + sfx, (slab, bits), _p(slab), _p(bits), B, S)
    return bits


def unpack_gf2(bits: torch.Tensor, S: int) -> torch.Tensor:
    """bit slab -> int8 slab of 0/1 values (tg_unpack_gf2); expand_states takes it on to float32."""
    B = _slab(bits, "bits", S, "_gf2").shape[0]
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
    sfx = _game_slab(slab, S)
    B = slab.shape[0]
    _operand(tape, "tape", torch.uint8, (B, layout(S).token_pitch))
    out = _slab(torch.empty_like(slab) if out is None else out, "out", S, sfx, B)
    flags = _operand(torch.empty(B, dtype=torch.uint8, device=slab.device) if flags is None else flags, "flags", torch.uint8, (B,))
    nnz = _operand(torch.empty(B, dtype=torch.int32, device=slab.device) if nnz is None else nnz, "nnz", torch.int32, (B,))
    _call("tg_step" + sfx, (slab, tape, out, flags, nnz,), _p(slab), _p(tape), _p(out), _p(flags), _p(nnz), B, S, shift)
    return out, flags, nnz


# ---------------------------------------------------------------- K2
def expand_children(slab: torch.Tensor, tape: torch.Tensor, S: int, shift: int, with_keys: bool = True):
    """Batched leaf expansion (tg_expand_children): children[b, c] = slab[b] - rank1(tape[b, c]).

    slab int8 or int16 (B, GP) (tg_expand_children_i16) or a bit slab (tg_expand_children_gf2), tape uint8 (B, k, TP).  Returns (children (B, k, GP) of the
    slab's dtype, flags (B, k), nnz (B, k), keys (B, k) or None).  Reference: act.py:266-275 get_child_states + the
    null / terminal / already-in-tree tests of extend_tree (act.py:177-195), for B states at once."""
    sfx = _game_slab(slab, S)
    B = slab.shape[0]
    k = _operand(tape, "tape", torch.uint8, (B, "k", layout(S).token_pitch)).shape[1]
    dev = slab.device
    children = torch.empty((B, k, slab.shape[1]), dtype=slab.dtype, device=dev)
    flags = torch.empty((B, k), dtype=torch.uint8, device=dev)
    nnz = torch.empty((B, k), dtype=torch.int32, device=dev)
    keys = torch.empty((B, k), dtype=torch.int64, device=dev) if with_keys else None
    _call("tg_expand_children" + sfx, (slab, tape, children, flags, nnz, keys,), _p(slab), _p(tape), k, _p(children), _p(flags), _p(nnz), _p(keys), B, S, shift)
    return children, flags, nnz, keys


def rollout(slab: torch.Tensor, tape: torch.Tensor, S: int, shift: int, out: torch.Tensor | None = None):
    """Apply a step-major tape (K, B, TP) to every game, freezing solved games.
    slab int8, int16 (tg_rollout_i16) or a bit slab (tg_rollout_gf2).  Returns (out, flags, nnz, steps).  Reference: datasets.py:144-153,
    training.py:336-342, act.py:49."""
    sfx = _game_slab(slab, S)
    B, tp = slab.shape[0], layout(S).token_pitch
    K = _operand(tape, "tape", torch.uint8, ("K", B, tp)).shape[0]
    out = _slab(torch.empty_like(slab) if out is None else out, "out", S, sfx, B)
    flags = torch.empty(B, dtype=torch.uint8, device=slab.device)
    nnz = torch.empty(B, dtype=torch.int32, device=slab.device)
    steps = torch.empty(B, dtype=torch.int32, device=slab.device)
    _call("tg_rollout" + sfx, (slab, tape, out, flags, nnz, steps,), _p(slab), _p(tape), B * tp, K, _p(out), _p(flags), _p(nnz), _p(steps), B, S, shift)
    return out, flags, nnz, steps


def replay(slab: torch.Tensor, tape: torch.Tensor, S: int, shift: int, out: torch.Tensor | None = None):
    """All K actions of a step-major tape applied without freezing (datasets.py:144-153); slab int8, int16
    (tg_replay_i16) or a bit slab (tg_replay_gf2).  Returns (out, flags, nnz)."""
    sfx = _game_slab(slab, S)
    B, tp = slab.shape[0], layout(S).token_pitch
    K = _operand(tape, "tape", torch.uint8, ("K", B, tp)).shape[0]
    out = _slab(torch.empty_like(slab) if out is None else out, "out", S, sfx, B)
    flags = torch.empty(B, dtype=torch.uint8, device=slab.device)
    nnz = torch.empty(B, dtype=torch.int32, device=slab.device)
    _call("tg_replay" + sfx, (slab, tape, out, flags, nnz,), _p(slab), _p(tape), B * tp, K, _p(out), _p(flags), _p(nnz), B, S, shift)
    return out, flags, nnz


# ---------------------------------------------------------------- K3
def _cat_arrays(values, probs):
    import numpy as np

    v = np.ascontiguousarray(values, dtype=np.int8)
    p = np.ascontiguousarray(probs, dtype=np.float64)
    if v.ndim != 1 or v.shape != p.shape or not 1 <= len(v) <= 8:
        raise TensorGameError("values/probs must be 1-D of equal length <= 8")
    return v, p


def _demos(name: str, n_demos: int, max_actions: int, S: int, box, values, probs, shift: int, seed: int, first_demo: int,
           device, max_tries: int, tape: torch.Tensor | None, slab: torch.Tensor | None, sfx: str):
    """The demo generators: the targets are an int8 slab (sfx "") or a bit slab ("_gf2"), and a box (nu, nv, nw) selects
    the box entry points.  tape and slab may be views into larger stores: the tape's steps at any stride."""
    tp = layout(S).token_pitch
    nu_nv_nw = () if box is None else _box_args(S, box)
    v, p = _cat_arrays(values, probs)
    dev = torch.device(device)
    if tape is None:
        tape = torch.empty((max_actions, n_demos, tp), dtype=torch.uint8, device=dev)
    _operand(tape, "tape", torch.uint8, (max_actions, n_demos, tp), rows=True)
    if slab is None:
        slab = torch.empty((n_demos, _game_pitch(sfx, S)), dtype=_SLAB_DTYPE[sfx], device=dev)
    _slab(slab, "bits" if sfx else "slab", S, sfx, n_demos)
    flags = torch.empty(n_demos, dtype=torch.uint8, device=dev)
    stride = tape.stride(0) if max_actions > 1 else n_demos * tp
    _call(name, (tape, slab, flags), seed, first_demo, n_demos, max_actions, S, *nu_nv_nw, shift, v.ctypes.data,
          p.ctypes.data, len(v), max_tries, _p(tape), stride, _p(slab), _p(flags))
    return tape, slab, flags


def make_synthetic_demos(n_demos: int, max_actions: int, S: int, values=(-1, 0, 1), probs=(0.15, 0.7, 0.15),
                         shift: int = 1, seed: int = 0, first_demo: int = 0, device="cuda", max_tries: int = 64,
                         tape: torch.Tensor | None = None, slab: torch.Tensor | None = None):
    """Throughput-mode demo generation (device Philox stream, tg_demo_gen_philox).

    Returns (tape uint8 (R, N, TP) step-major, slab int8 (N, GP), flags uint8 (N,)).
    Same distribution and rejection rule as utils.py:203-233; NOT the torch RNG stream --
    use demos_from_seed for same-seed parity with the reference."""
    return _demos("tg_demo_gen_philox", n_demos, max_actions, S, None, values, probs, shift, seed, first_demo, device,
                  max_tries, tape, slab, "")


def make_synthetic_demos_gf2(n_demos: int, max_actions: int, S: int, values=(-1, 0, 1), probs=(0.15, 0.7, 0.15), shift: int = 1,
                             seed: int = 0, first_demo: int = 0, device="cuda", max_tries: int = 64, tape: torch.Tensor | None = None,
                             bits: torch.Tensor | None = None):
    """Throughput-mode demo generation modulo 2 (tg_demo_gen_gf2): every factor has an odd entry, so no term vanishes mod 2,
    and the targets are bit slabs (the xor of the terms), written without an int8 slab.

    Returns (tape uint8 (R, N, TP) step-major, bits int32 (N, GB/4), flags uint8 (N,): TG_FLAG_EXHAUSTED or 0).  Where 0
    is the only even value of the alphabet, the tape is make_synthetic_demos' for the same arguments and the bits are
    pack_gf2 of its targets."""
    return _demos("tg_demo_gen_gf2", n_demos, max_actions, S, None, values, probs, shift, seed, first_demo, device,
                  max_tries, tape, bits, "_gf2")


# ---------------------------------------------------------------- rectangular products <n, m, p>
_SIZES = (4, 9, 16, 25)


def matmul_box(n: int, m: int, p: int) -> tuple[int, tuple[int, int, int]]:
    """<n, m, p> (A n x m, B m x p, C n x p) is a tensor of shape box = (n m, m p, n p).  Returns (S, box): the smallest
    game size S in {4, 9, 16, 25} that holds every mode of the box.  Raises for a box with a mode beyond 25."""
    if min(n, m, p) < 1:
        raise TensorGameError(f"<{n}, {m}, {p}>: sizes must be >= 1")
    box = (n * m, m * p, n * p)
    for S in _SIZES:
        if max(box) <= S:
            return S, box
    raise TensorGameError(f"<{n}, {m}, {p}>: its box {box} does not fit the largest game size 25")


def matmul_tensor(n: int, m: int, p: int, S: int | None = None) -> torch.Tensor:
    """The matrix multiplication tensor of <n, m, p> zero-padded to (S, S, S), int8 on the host (S defaults to
    matmul_box's): T[i m + j][j p + k][i p + k] = 1 for i < n, j < m, k < p, the reference's convention with the C index
    not transposed.  At n = m = p it is utils.build_matmul_tensor(1, n, n, n)[0].  pack_states, pack_states16 and
    pack_gf2 turn it into any slab format; its float() is a start_tensor for TensorGameDataset.  Every factorization of
    the padded tensor, truncated to the box (project_to_box), is one of <n, m, p> with at most as many non-null terms."""
    S0, box = matmul_box(n, m, p)
    S = S0 if S is None else S
    if S not in _SIZES or S < S0:
        raise TensorGameError(f"<{n}, {m}, {p}> needs S in {tuple(s for s in _SIZES if s >= S0)}, got {S}")
    T = torch.zeros((S, S, S), dtype=torch.int8)
    i, j, k = torch.meshgrid(torch.arange(n), torch.arange(m), torch.arange(p), indexing="ij")
    T[i * m + j, j * p + k, i * p + k] = 1
    return T


def _box_args(S: int, box) -> tuple[int, int, int]:
    nu, nv, nw = (int(x) for x in box)
    if not all(1 <= x <= S for x in (nu, nv, nw)):
        raise TensorGameError(f"box {tuple(box)} must lie in [1, {S}]^3")
    return nu, nv, nw


def make_synthetic_demos_box(n_demos: int, max_actions: int, S: int, box, values=(-1, 0, 1), probs=(0.15, 0.7, 0.15),
                             shift: int = 1, seed: int = 0, first_demo: int = 0, device="cuda", max_tries: int = 64,
                             tape: torch.Tensor | None = None, slab: torch.Tensor | None = None):
    """make_synthetic_demos with every factor confined to box = (nu, nv, nw) (tg_demo_gen_box, contract box v1): the
    demonstrations of a rectangular product played at size S (matmul_box).  Every entry of u beyond nu, of v beyond nv and
    of w beyond nw is 0, and each factor has a non-zero entry inside the box.  With the full box (S, S, S) it is contract
    v1 at S.  The targets are what accumulate_demos writes for the tape; beyond int8 re-sum with accumulate_demos16.

    Returns (tape uint8 (R, N, TP) step-major, slab int8 (N, GP), flags uint8 (N,): FLAG_EXHAUSTED | FLAG_RANGE).  tape
    and slab may be views into larger stores (several shapes in one S = 25 store: one call per shape into slices, with
    disjoint first_demo ranges)."""
    return _demos("tg_demo_gen_box", n_demos, max_actions, S, box, values, probs, shift, seed, first_demo, device,
                  max_tries, tape, slab, "")


def make_synthetic_demos_box_gf2(n_demos: int, max_actions: int, S: int, box, values=(-1, 0, 1), probs=(0.15, 0.7, 0.15),
                                 shift: int = 1, seed: int = 0, first_demo: int = 0, device="cuda", max_tries: int = 64,
                                 tape: torch.Tensor | None = None, bits: torch.Tensor | None = None):
    """make_synthetic_demos_gf2 with every factor confined to box = (nu, nv, nw) (tg_demo_gen_box_gf2, contract box v1
    mod 2: each factor has an odd entry inside the box).  Returns (tape uint8 (R, N, TP), bits int32 (N, GB/4), flags
    uint8 (N,): FLAG_EXHAUSTED or 0)."""
    return _demos("tg_demo_gen_box_gf2", n_demos, max_actions, S, box, values, probs, shift, seed, first_demo, device,
                  max_tries, tape, bits, "_gf2")


def box_bases(mats: torch.Tensor, box) -> torch.Tensor:
    """Change-of-basis triples that keep the box: matrix f keeps its leading box[f] x box[f] block and is the identity
    elsewhere, so entries outside the box stay zero and factors inside it stay inside.  mats int8 (N, 3, S, S)
    (sample_unimodular, S <= 16) or GF(2) bit matrices int32 (N, 3, S) (sample_invertible_gf2; word r = row r, bit c =
    entry (r, c)).  Both samplers draw M = L U (L unit lower, U upper triangular): the leading k x k block is L11 U11,
    unimodular (invertible over GF(2)) and distributed as the sampler's own draw at size k, so the results are unimodular
    (invertible) and their inverses are the block-diagonal inverses invert_bases(_gf2) return."""
    bits = mats.dtype == torch.int32
    S = mats.shape[-1]
    m = mats.reshape((-1, 3, S) if bits else (-1, 3, S, S)).clone()
    dev = mats.device
    r = torch.arange(S, device=dev)
    for f in range(3):
        k = _box_args(S, box)[f]
        if bits:
            # rows < k keep their bits < k; rows >= k are unit rows
            keep = torch.where(r < k, (1 << k) - 1, 0).to(torch.int32)
            unit = torch.where(r < k, 0, torch.bitwise_left_shift(torch.ones_like(r), r)).to(torch.int32)
            m[:, f] = (m[:, f] & keep) | unit
        else:
            inside = (r[:, None] < k) & (r[None, :] < k)
            eye = torch.eye(S, dtype=torch.int8, device=dev)
            m[:, f] = torch.where(inside, m[:, f], eye)
    return m


def project_to_box(tape: torch.Tensor, S: int, box, shift: int) -> torch.Tensor:
    """The projection onto the box of every action of a tape (..., TP): tokens of u beyond box[0], of v beyond box[1]
    and of w beyond box[2] become `shift` (the coefficient 0).  The projection is linear and fixes every tensor that is
    zero outside the box, so a tape that sums to such a target still sums to it afterwards.  Returns a new tape."""
    _device(_operand(tape, "tape", torch.uint8))
    nu, nv, nw = _box_args(S, box)
    e = torch.arange(S, device=tape.device)
    out = torch.cat([(e >= n) for n in (nu, nv, nw)])
    res = tape.clone()
    res[..., : 3 * S][..., out] = shift
    return res


def _accumulate(name: str, tape: torch.Tensor, S: int, shift: int, slab: torch.Tensor | None, slab_name: str, sfx: str):
    """The accumulate_demos entry points: the sum of a step-major tape (R, N, TP) into an int8 ("") or int16 ("_i16")
    slab."""
    tp = layout(S).token_pitch
    R, N = _operand(tape, "tape", torch.uint8, ("R", "N", tp)).shape[:2]
    if slab is None:
        slab = torch.empty((N, layout(S).game_pitch), dtype=_SLAB_DTYPE[sfx], device=tape.device)
    _slab(slab, slab_name, S, sfx, N)
    flags = torch.empty(N, dtype=torch.uint8, device=tape.device)
    _call(name, (tape, slab, flags), _p(tape), N * tp, N, R, S, shift, _p(slab), _p(flags))
    return slab, flags


def accumulate_demos(tape: torch.Tensor, S: int, shift: int, slab: torch.Tensor | None = None):
    """slab[n] = sum_r rank1(tape[r, n]) (tg_demo_accumulate).  Returns (slab, flags)."""
    return _accumulate("tg_demo_accumulate", tape, S, shift, slab, "slab", "")


def accumulate_demos16(tape: torch.Tensor, S: int, shift: int, slab16: torch.Tensor | None = None):
    """The same sum as accumulate_demos into an int16 slab (tg_demo_accumulate_i16): exact for every tape; the flag
    says an entry does not fit int16.  Where targets beyond the int8 slab's zone go (the reference accumulates them in
    float32 without limit, utils.py:218-232).  Returns (slab16 int16 (N, GP), flags)."""
    return _accumulate("tg_demo_accumulate_i16", tape, S, shift, slab16, "slab16", "_i16")


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
    _call("tg_demo_from_ustream", (u, tape, slab, flags, result, ws,), _p(u), n_u, v.ctypes.data, p.ctypes.data, len(v), max_actions, S,
          shift, n_demos, _p(tape), n_demos * lay.token_pitch, _p(slab), _p(flags), _p(result), _p(ws), ws_bytes)
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
    return _accumulate("tg_demo_accumulate_tc", tape, 16, shift, slab, "slab", "")


# ---------------------------------------------------------------- K4 / K6 / K7
def _sample_outputs(idx: torch.Tensor, dim_t: int, S: int, dev) -> tuple:
    """The outputs of the sample batchers for the indices idx: states f32 (nb,dim_t,S,S,S), scalars f32 (nb,1), actions
    i64 (nb,3S), rewards f32 (nb,1)."""
    nb = _operand(idx, "idx", torch.int64).numel()
    return (torch.empty((nb, dim_t, S, S, S), dtype=torch.float32, device=dev), torch.empty((nb, 1), dtype=torch.float32, device=dev),
            torch.empty((nb, 3 * S), dtype=torch.int64, device=dev), torch.empty((nb, 1), dtype=torch.float32, device=dev))


def demo_samples(tape: torch.Tensor, slab: torch.Tensor, idx: torch.Tensor, S: int, dim_t: int, replay_shift: int = 1):
    """Batch of SyntheticDemoDataset.__getitem__ results (datasets.py:77-122) from the in-HBM demo store.
    Returns (states f32 (nb,dim_t,S,S,S), scalars f32 (nb,1), actions i64 (nb,3S), rewards f32 (nb,1))."""
    tp = layout(S).token_pitch
    R, N = _operand(tape, "tape", torch.uint8, ("R", "N", tp)).shape[:2]
    _slab(slab, "slab", S, "", N)
    out = _sample_outputs(idx, dim_t, S, tape.device)
    _call("tg_demo_sample", (tape, slab, idx, *out), _p(tape), N * tp, _p(slab), N, R, S, dim_t, replay_shift, _p(idx),
          idx.numel(), *map(_p, out))
    return out


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
        N = _operand(records, "records", torch.uint8, ("N", "R", layout(S).token_pitch)).shape[0]
        targets = targets.contiguous()
        self.bits = _game_slab(targets, S, "targets", N) == "_gf2"
        _device(records, targets)
        self.records, self.targets, self.S, self.shift = records, targets, S, shift
        self.N, self.R = records.shape[0], records.shape[1]
        if self.bits:
            target_bound = 0
        elif target_bound is None:
            target_bound = 127 if targets.dtype == torch.int8 else (int(targets.abs().max()) if self.N else 0)
        self.target_bound = int(target_bound)

    @classmethod
    def from_tape(cls, tape: torch.Tensor, targets: torch.Tensor, S: int, shift: int) -> "DemoStore":
        """From a step-major tape (R, N, TP) (tg_tape_to_demo_major) and its target slab."""
        tp = layout(S).token_pitch
        R, N = _operand(tape, "tape", torch.uint8, ("R", "N", tp)).shape[:2]
        records = torch.empty((N, R, tp), dtype=torch.uint8, device=tape.device)
        _call("tg_tape_to_demo_major", (tape, records), _p(tape), N * tp, _p(records), N, R, S)
        return cls(records, targets, S, shift)

    def tape(self) -> torch.Tensor:
        """The step-major view (R, N, TP) of the records (a strided view, no copy)."""
        return self.records.transpose(0, 1)

    def samples(self, idx: torch.Tensor, dim_t: int, replay_shift: int = 1):
        """Batch of SyntheticDemoDataset.__getitem__ results (datasets.py:77-122) for sample indices demo * R + action
        (tg_demo_sample_dm; with bit targets tg_demo_sample_gf2, states mod 2 as 0/1).  Returns (states f32
        (nb,dim_t,S,S,S), scalars f32 (nb,1), actions i64 (nb,3S), rewards f32 (nb,1))."""
        out = _sample_outputs(idx, dim_t, self.S, self.records.device)
        operands = (self.records, self.targets, idx, *out)
        outputs = (_p(idx), idx.numel(), *map(_p, out))
        if self.bits:
            _call("tg_demo_sample_gf2", operands, _p(self.records), _p(self.targets), self.N, self.R, self.S, dim_t, replay_shift, *outputs)
        else:
            _call("tg_demo_sample_dm", operands, _p(self.records), _p(self.targets), int(self.targets.dtype == torch.int16),
                  self.target_bound, self.N, self.R, self.S, dim_t, replay_shift, *outputs)
        return out


def slice_rank(slab: torch.Tensor, S: int) -> torch.Tensor:
    """get_rank per game (utils.py:134-140) of an int8 or int16 slab (tg_slice_rank_i16): int32 (B,).  Of a bit slab
    (tg_slice_rank_gf2): the sum of the slices' ranks over GF(2)."""
    sfx = _game_slab(slab, S)
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
    sfx = _game_slab(slab, S)
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
    _call("tg_sample_unimodular", (mats,), seed, first, n, S, float(p_nonzero), _p(mats))
    return mats


def _bases(mats: torch.Tensor, S: int, N: int, gf2: bool) -> tuple[torch.Tensor, int]:
    """The (A, B, C) triples of a change of basis of N games, one per game or one shared: int8 (N or 1, 3, S, S), or
    bit matrices int32 (N or 1, 3, S) over GF(2).  Returns them in that shape and the entry points' per_game."""
    tail = (3, S) if gf2 else (3, S, S)
    _operand(mats, "mats", torch.int32 if gf2 else torch.int8)
    one = math.prod(tail)
    if mats.numel() not in (one, N * one):
        raise TensorGameError("mats must hold one (A,B,C) triple or one per game")
    m = mats if mats.shape[1:] == tail else mats.view(-1, *tail)
    return m, int(m.shape[0] == N and N > 1)


def _factors(tape: torch.Tensor, m: torch.Tensor, per_game: int, S: int, shift: int, shift_out: int | None,
             flags: torch.Tensor | None = None, skip_empty: bool = True) -> torch.Tensor:
    """u' = A u, v' = B v, w' = C w for every record of a checked step-major tape (R, N, TP): over Z with flags
    (tg_change_of_basis_factors), over GF(2) without (tg_change_of_basis_factors_gf2).  A tape without records is
    returned without a launch unless skip_empty is False (the entry points refuse R = 0)."""
    R, N, tp = tape.shape
    tape_out = torch.empty_like(tape)
    if R == 0 and skip_empty:
        _device(tape, m, flags)  # no launch, and still no CPU path
        return tape_out
    shift_out = shift if shift_out is None else shift_out
    if flags is None:
        _call("tg_change_of_basis_factors_gf2", (tape, m, tape_out), _p(tape), N * tp, shift, _p(m), per_game, _p(tape_out),
              N * tp, shift_out, N, R, S)
    else:
        _call("tg_change_of_basis_factors", (tape, m, tape_out, flags), _p(tape), N * tp, shift, _p(m), per_game, _p(tape_out),
              N * tp, shift_out, _p(flags), N, R, S)
    return tape_out


def change_of_basis(slab: torch.Tensor, mats: torch.Tensor, S: int, tape: torch.Tensor | None = None, shift: int = 0,
                    shift_out: int | None = None, out: torch.Tensor | None = None, out_dtype: torch.dtype = torch.int8,
                    return_path_stats: bool = False):
    """T' = T x1 A x2 B x3 C (and u' = A u, v' = B v, w' = C w for a step-major tape).

    mats int8 (N, 3, S, S) per game or (1, 3, S, S) / (3, S, S) shared.  The result is an int8 slab (flag RANGE: an
    entry left [-64, 63]) or, with out_dtype / out of torch.int16, an int16 slab (SURVEY 8(d)'s format; flag RANGE: an
    entry does not fit int16).  Returns (slab', flags) or (slab', tape', flags); with return_path_stats a dict counting
    the games per kernel path is appended.  Not in the reference: AlphaTensor paper, Methods "Change of basis"."""
    N = _slab(slab, "slab", S, "").shape[0]
    m, per_game = _bases(mats, S, N, False)
    if out is None:
        out = torch.empty(slab.shape, dtype=out_dtype, device=slab.device)
    sfx = "_i16" if getattr(out, "dtype", None) == torch.int16 else ""
    _slab(out, "out", S, sfx, N)
    if tape is not None:
        _operand(tape, "tape", torch.uint8, ("R", N, layout(S).token_pitch))
    flags = torch.zeros(N, dtype=torch.uint8, device=slab.device)
    _call("tg_change_of_basis" + sfx, (slab, m, out, flags), _p(slab), _p(m), per_game, _p(out), _p(flags), N, S)
    stats = None
    if return_path_stats:
        exact = int(((flags & FLAG_PATH_EXACT) != 0).sum().item())
        planes = int(((flags & FLAG_PATH_PLANES) != 0).sum().item())
        stats = {"games": N, "fast_path": N - exact - planes, "byte_plane_path": planes, "exact_int32_redo": exact}
    if tape is None:
        return (out, flags, stats) if return_path_stats else (out, flags)
    tape_out = _factors(tape, m, per_game, S, shift, shift_out, flags, skip_empty=False)
    return (out, tape_out, flags, stats) if return_path_stats else (out, tape_out, flags)


def change_of_basis_factors(tape: torch.Tensor, mats: torch.Tensor, S: int, shift: int, shift_out: int | None = None):
    """u' = A u, v' = B v, w' = C w for every record of a step-major tape (R, N, TP), without a slab
    (tg_change_of_basis_factors): coefficients are token - shift, tokens out are coefficient + shift_out (default shift,
    in [1, 127]).  mats int8 (N, 3, S, S) per game or (1, 3, S, S) / (3, S, S) shared.  Returns (tape', flags uint8
    (N,)): FLAG_TOKEN_RANGE where a transformed entry left [-shift_out, shift_out].  With the triples of invert_bases this
    maps factors found in a changed basis back to the original one."""
    N = _operand(tape, "tape", torch.uint8, ("R", "N", layout(S).token_pitch)).shape[1]
    m, per_game = _bases(mats, S, N, False)
    flags = torch.zeros(N, dtype=torch.uint8, device=tape.device)
    return _factors(tape, m, per_game, S, shift, shift_out, flags), flags


def _invert(mats: torch.Tensor, out: torch.Tensor | None, gf2: bool):
    """invert_bases (int8 (N, 3, S, S)) and invert_bases_gf2 (bit matrices int32 (N, 3, S))."""
    S = mats.shape[-1]
    tail, dtype = ((3, S), torch.int32) if gf2 else ((3, S, S), torch.int8)
    _operand(mats, "mats", dtype)
    if mats.dim() not in (len(tail), len(tail) + 1) or mats.shape[-len(tail):] != tail:
        dims = ", ".join(("3", "S", "S")[:len(tail)])
        raise TensorGameError(f"mats must be (N, {dims}) or ({dims})")
    m = mats.view(-1, *tail)
    out = _operand(torch.empty_like(m) if out is None else out, "out", dtype)
    if out.numel() != m.numel():
        raise TensorGameError("out must hold as many matrices as mats")
    out = out.view(m.shape)
    flags = torch.empty(m.shape[0], dtype=torch.uint8, device=mats.device)
    _call("tg_invert_bases_gf2" if gf2 else "tg_invert_bases", (m, out, flags), _p(m), _p(out), _p(flags), m.shape[0], S)
    return out, flags


def invert_bases(mats: torch.Tensor, out: torch.Tensor | None = None):
    """The inverse of every matrix of (A, B, C) triples over Z (tg_invert_bases): mats int8 (N, 3, S, S), or (3, S, S) as
    N = 1, S in {4, 9, 16}.  Returns (inv int8 (N, 3, S, S), flags uint8 (N,)): inv[n, f] is the integer inverse of
    mats[n, f] where one exists with every entry in [-128, 127]; otherwise that matrix is all zeros and flags[n] =
    FLAG_SINGULAR.  out may be mats (in place)."""
    return _invert(mats, out, False)


# ---------------------------------------------------------------- K5 mod 2
def sample_invertible_gf2(n: int, S: int, seed: int = 0, first: int = 0, p_nonzero: float = 0.3, device="cuda") -> torch.Tensor:
    """Random (A, B, C) per game, each invertible over GF(2), as bit matrices int32 (n, 3, S): word r of a matrix is its
    row r, bit c its entry (r, c) (tg_sample_invertible_gf2).  At S <= 16 these are sample_unimodular(n, S, seed, first,
    p_nonzero) mod 2."""
    dev = torch.device(device)
    if dev.type != "cuda":
        raise TensorGameError("sample_invertible_gf2 needs a CUDA device (there is no CPU path)")
    mats = torch.empty((n, 3, S), dtype=torch.int32, device=dev)
    _call("tg_sample_invertible_gf2", (mats,), seed, first, n, S, float(p_nonzero), _p(mats))
    return mats


def change_of_basis_gf2(bits: torch.Tensor, mats: torch.Tensor, S: int, tape: torch.Tensor | None = None, shift: int = 1,
                        shift_out: int | None = None, out: torch.Tensor | None = None):
    """T' = T x1 A x2 B x3 C over GF(2) on a bit slab (tg_change_of_basis_gf2), and u' = A u, v' = B v, w' = C w mod 2
    for a step-major tape (R, N, TP) (tg_change_of_basis_factors_gf2: tokens read with `shift`, written as residue +
    shift_out, default shift).  mats: bit matrices int32 (N, 3, S) per game, or (1, 3, S) / (3, S) shared.  out may be
    bits (in place).  Returns bits', or (bits', tape') when a tape is given.  Nothing can leave the format mod 2, so there
    are no flags.  Not in the reference: AlphaTensor paper, Methods "Change of basis", in modular arithmetic."""
    N = _slab(bits, "bits", S, "_gf2").shape[0]
    m, per_game = _bases(mats, S, N, True)
    out = _slab(torch.empty_like(bits) if out is None else out, "out", S, "_gf2", N)
    if tape is not None:
        _operand(tape, "tape", torch.uint8, ("R", N, layout(S).token_pitch))
    _call("tg_change_of_basis_gf2", (bits, m, out), _p(bits), _p(m), per_game, _p(out), N, S)
    if tape is None:
        return out
    return out, _factors(tape, m, per_game, S, shift, shift_out)


def change_of_basis_factors_gf2(tape: torch.Tensor, mats: torch.Tensor, S: int, shift: int = 1, shift_out: int | None = None):
    """u' = A u, v' = B v, w' = C w mod 2 for every record of a step-major tape (R, N, TP), without a bit slab
    (tg_change_of_basis_factors_gf2): tokens read with `shift`, written as residue + shift_out (default shift), both in
    [1, 4].  mats: bit matrices int32 (N, 3, S) per game, or (1, 3, S) / (3, S) shared.  Returns tape'."""
    N = _operand(tape, "tape", torch.uint8, ("R", "N", layout(S).token_pitch)).shape[1]
    m, per_game = _bases(mats, S, N, True)
    return _factors(tape, m, per_game, S, shift, shift_out)


def invert_bases_gf2(mats: torch.Tensor, out: torch.Tensor | None = None):
    """The inverse over GF(2) of every matrix of bit-matrix triples (tg_invert_bases_gf2): mats int32 (N, 3, S), or (3, S)
    as N = 1, S in {4, 9, 16, 25}; bits S to 31 of a row are ignored.  Returns (inv int32 (N, 3, S), flags uint8 (N,)):
    a matrix singular over GF(2) comes back as zero rows with flags[n] = FLAG_SINGULAR.  out may be mats (in place)."""
    return _invert(mats, out, True)


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
    inside the C library (tg_step_host).

    step and rollout take int8 slabs (B, GP), int16 slabs (B, GP) or int32 bit slabs (B, GB/4) and dispatch on the
    dtype as step_batch does (tg_step_host, tg_step_host_i16, tg_step_host_gf2); make_demos takes an int8 slab or an
    int32 bit slab for the targets.  One context serves every format; the first int16 call doubles its slab staging."""

    def __init__(self, S: int, device: int = 0, chunk: int = 1 << 16):
        self.S, self.lay = S, layout(S)
        self._ctx = C.c_void_p()
        check(_lib.lib().tg_host_ctx_create(C.byref(self._ctx), device, S, chunk), "tg_host_ctx_create")

    def _format(self, slab: torch.Tensor, out: torch.Tensor, records: torch.Tensor, steps: bool, flags: torch.Tensor,
                *int32s: torch.Tensor) -> str:
        """The entry-point suffix of a call ("", "_i16" or "_gf2") after checking its CPU tensors, before the context is
        used: slab and out of one format, (B, GP) or (B, GB/4); records uint8 (B, TP) or, with steps, a step-major tape
        (K, B, TP); flags uint8 (B,) and the int32 per-game arrays (nnz, steps) (B,)."""
        for t in (slab, out, records, flags, *int32s):
            if getattr(t, "is_cuda", False):
                raise TensorGameError("HostStepper takes CPU tensors")
        sfx = _game_slab(slab, self.S)
        B = slab.shape[0]
        _slab(out, "out", self.S, sfx, B)
        _operand(records, "tape", torch.uint8, ("K",) * steps + (B, self.lay.token_pitch))
        _operand(flags, "flags", torch.uint8, (B,))
        for name, t in zip(("nnz", "steps"), int32s):
            _operand(t, name, torch.int32, (B,))
        return sfx

    def step(self, slab: torch.Tensor, tape: torch.Tensor, out: torch.Tensor, flags: torch.Tensor, nnz: torch.Tensor,
             shift: int) -> None:
        name = "tg_step_host" + self._format(slab, out, tape, False, flags, nnz)
        check(getattr(_lib.lib(), name)(self._ctx, _p(slab), _p(tape), _p(out), _p(flags), _p(nnz), slab.shape[0], shift), name)

    def rollout(self, slab: torch.Tensor, tape: torch.Tensor, out: torch.Tensor, flags: torch.Tensor, nnz: torch.Tensor,
                steps: torch.Tensor, shift: int) -> None:
        """K fused steps per PCIe round trip (tg_rollout_host): tape is the dense step-major CPU tape (K, B, TP)."""
        name = "tg_rollout_host" + self._format(slab, out, tape, True, flags, nnz, steps)
        check(getattr(_lib.lib(), name)(self._ctx, _p(slab), _p(tape), tape.shape[0], _p(out), _p(flags), _p(nnz), _p(steps),
                                        slab.shape[0], shift), name)

    def make_demos(self, tape: torch.Tensor, slab: torch.Tensor, flags: torch.Tensor, shift: int, values, probs, seed: int = 0,
                   first_demo: int = 0, max_tries: int = 64) -> None:
        """Synthetic demonstrations straight into CPU buffers (tg_demo_gen_host): tape (R, N, TP), slab (N, GP), flags (N,).
        An int32 bit slab (N, GB/4) takes the demos modulo 2 (tg_demo_gen_host_gf2, the demos of make_synthetic_demos_gf2)."""
        sfx = self._format(slab, slab, tape, True, flags)
        if sfx == "_i16":
            raise TensorGameError("HostStepper.make_demos writes int8 slabs or int32 bit slabs, not int16 targets")
        v, p = _cat_arrays(values, probs)
        name = "tg_demo_gen_host" + sfx
        check(getattr(_lib.lib(), name)(self._ctx, seed, first_demo, slab.shape[0], tape.shape[0], shift, v.ctypes.data,
                                        p.ctypes.data, len(v), max_tries, _p(tape), _p(slab), _p(flags)), name)

    def close(self) -> None:
        if self._ctx:
            _lib.lib().tg_host_ctx_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
