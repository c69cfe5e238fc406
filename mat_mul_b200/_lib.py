"""Loader for libtensorgame_b200.so (the C-ABI CUDA library, include/tensorgame.h).

The library is built in-tree with nvcc for sm_100a only.  There is no CPU
fallback: if the library cannot be loaded, every compute entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
# TG_TUNING=1 selects the sweep build (-DTG_TUNING: extra kernel instantiations, getenv knobs, tg_tune_* entry points);
# the production library has none of them
TUNING = os.environ.get("TG_TUNING", "0") not in ("", "0")
LIB_PATH = PKG / ("libtensorgame_b200_tuning.so" if TUNING else "libtensorgame_b200.so")
HASH_PATH = LIB_PATH.with_suffix(".srchash")
HEADER = PKG.parent / "include" / "tensorgame.h"

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared", "--threads", "0",
]

TG_OK = 0
FLAG_TERMINAL = 1
FLAG_NULL = 2
FLAG_RANGE = 4
FLAG_EXHAUSTED = 8
FLAG_TOKEN_RANGE = 16
FLAG_PATH_PLANES = 32
FLAG_PATH_EXACT = 64
FLAG_SINGULAR = 128


class TensorGameError(RuntimeError):
    pass


def sources() -> list[Path]:
    return sorted(CSRC.glob("*.cu"))


def _source_hash() -> str:
    """Content hash of everything the library is built from (sources, header, flags): unlike mtimes it survives the
    copy to the GPU box, so a shipped .so is recognised as current there and a stale one is recognised as stale."""
    import hashlib

    h = hashlib.sha256(" ".join(NVCC_FLAGS + (["-DTG_TUNING"] if TUNING else [])).encode())
    for d in sorted(list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh"))) + [HEADER]:
        h.update(d.name.encode())
        h.update(d.read_bytes())
    return h.hexdigest()


def _stale() -> bool:
    if not LIB_PATH.exists() or not HASH_PATH.exists():
        return True
    return HASH_PATH.read_text().strip() != _source_hash()


def header_version() -> int:
    import re

    return int(re.search(r"#define\s+TG_VERSION\s+(\d+)", HEADER.read_text()).group(1))


def build(force: bool = False, verbose: bool = False) -> Path:
    """nvcc -gencode arch=compute_100a,code=sm_100a ... -> mat_mul_b200/libtensorgame_b200.so"""
    if not force and not _stale():
        return LIB_PATH
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc, *NVCC_FLAGS, *(["-DTG_TUNING"] if TUNING else []), "-o", str(LIB_PATH), *map(str, sources())]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    digest = _source_hash()
    HASH_PATH.unlink(missing_ok=True)
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise TensorGameError(f"nvcc failed:\n{' '.join(cmd)}\n{res.stdout}\n{res.stderr}")
    HASH_PATH.write_text(digest + "\n")
    if verbose:
        print(res.stderr)
    return LIB_PATH


_lib = None

_i8p = C.c_void_p
_vp = C.c_void_p

_SIGNATURES = {
    "tg_version": (C.c_int, []),
    "tg_last_cuda_error": (C.c_int, []),
    "tg_error_string": (C.c_char_p, [C.c_int]),
    "tg_layout": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "tg_pack_f32": (C.c_int, [_vp, C.c_int64, _vp, C.c_int64, C.c_int, _vp, _vp]),
    "tg_expand_f32": (C.c_int, [_vp, _vp, C.c_int64, C.c_int64, C.c_int, _vp]),
    "tg_pack_actions_i64": (C.c_int, [_vp, _vp, C.c_int64, C.c_int, _vp, _vp]),
    "tg_unpack_actions_i64": (C.c_int, [_vp, _vp, C.c_int64, C.c_int, _vp]),
    "tg_step": (C.c_int, [_vp, _vp, _vp, _vp, _vp, C.c_int64, C.c_int, C.c_int, _vp]),
    "tg_expand_children": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, _vp, _vp, C.c_int64, C.c_int, C.c_int, _vp]),
    "tg_rollout": (C.c_int, [_vp, _vp, C.c_int64, C.c_int, _vp, _vp, _vp, _vp, C.c_int64, C.c_int, C.c_int, _vp]),
    "tg_replay": (C.c_int, [_vp, _vp, C.c_int64, C.c_int, _vp, _vp, _vp, C.c_int64, C.c_int, C.c_int, _vp]),
    "tg_demo_gen_philox": (C.c_int, [C.c_uint64, C.c_uint64, C.c_int64, C.c_int, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_int,
                                     _vp, C.c_int64, _vp, _vp, _vp]),
    "tg_demo_alias_tables": (C.c_int, [_vp, _vp, C.c_int, C.c_int, _vp]),
    "tg_demo_accumulate": (C.c_int, [_vp, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int, _vp, _vp, _vp]),
    "tg_demo_accumulate_tc": (C.c_int, [_vp, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int, _vp, _vp, _vp]),
    "tg_demo_sample": (C.c_int, [_vp, C.c_int64, _vp, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, _vp, C.c_int64, _vp, _vp, _vp,
                                 _vp, _vp]),
    "tg_demo_sample_dm": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, _vp, C.c_int64, _vp,
                                    _vp, _vp, _vp, _vp]),
    "tg_tape_to_demo_major": (C.c_int, [_vp, C.c_int64, _vp, C.c_int64, C.c_int, C.c_int, _vp]),
    "tg_slice_rank": (C.c_int, [_vp, _vp, C.c_int64, C.c_int, _vp]),
    "tg_state_key": (C.c_int, [_vp, _vp, C.c_int64, C.c_int, _vp]),
    "tg_change_of_basis": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, C.c_int64, C.c_int, _vp]),
    "tg_change_of_basis_i16": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, C.c_int64, C.c_int, _vp]),
    "tg_demo_accumulate_i16": (C.c_int, [_vp, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int, _vp, _vp, _vp]),
    "tg_pack_f32_i16": (C.c_int, [_vp, C.c_int64, _vp, C.c_int64, C.c_int, _vp, _vp]),
    "tg_expand_f32_i16": (C.c_int, [_vp, _vp, C.c_int64, C.c_int64, C.c_int, _vp]),
    "tg_step_i16": (C.c_int, [_vp, _vp, _vp, _vp, _vp, C.c_int64, C.c_int, C.c_int, _vp]),
    "tg_expand_children_i16": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, _vp, _vp, C.c_int64, C.c_int, C.c_int, _vp]),
    "tg_rollout_i16": (C.c_int, [_vp, _vp, C.c_int64, C.c_int, _vp, _vp, _vp, _vp, C.c_int64, C.c_int, C.c_int, _vp]),
    "tg_replay_i16": (C.c_int, [_vp, _vp, C.c_int64, C.c_int, _vp, _vp, _vp, C.c_int64, C.c_int, C.c_int, _vp]),
    "tg_state_key_i16": (C.c_int, [_vp, _vp, C.c_int64, C.c_int, _vp]),
    "tg_slice_rank_i16": (C.c_int, [_vp, _vp, C.c_int64, C.c_int, _vp]),
    "tg_layout_gf2": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "tg_pack_gf2": (C.c_int, [_vp, _vp, C.c_int64, C.c_int, _vp]),
    "tg_pack_gf2_i16": (C.c_int, [_vp, _vp, C.c_int64, C.c_int, _vp]),
    "tg_unpack_gf2": (C.c_int, [_vp, _vp, C.c_int64, C.c_int, _vp]),
    "tg_step_gf2": (C.c_int, [_vp, _vp, _vp, _vp, _vp, C.c_int64, C.c_int, C.c_int, _vp]),
    "tg_expand_children_gf2": (C.c_int, [_vp, _vp, C.c_int, _vp, _vp, _vp, _vp, C.c_int64, C.c_int, C.c_int, _vp]),
    "tg_rollout_gf2": (C.c_int, [_vp, _vp, C.c_int64, C.c_int, _vp, _vp, _vp, _vp, C.c_int64, C.c_int, C.c_int, _vp]),
    "tg_replay_gf2": (C.c_int, [_vp, _vp, C.c_int64, C.c_int, _vp, _vp, _vp, C.c_int64, C.c_int, C.c_int, _vp]),
    "tg_state_key_gf2": (C.c_int, [_vp, _vp, C.c_int64, C.c_int, _vp]),
    "tg_slice_rank_gf2": (C.c_int, [_vp, _vp, C.c_int64, C.c_int, _vp]),
    "tg_change_of_basis_gf2": (C.c_int, [_vp, _vp, C.c_int, _vp, C.c_int64, C.c_int, _vp]),
    "tg_change_of_basis_factors_gf2": (C.c_int, [_vp, C.c_int64, C.c_int, _vp, C.c_int, _vp, C.c_int64, C.c_int, C.c_int64, C.c_int,
                                                 C.c_int, _vp]),
    "tg_sample_invertible_gf2": (C.c_int, [C.c_uint64, C.c_uint64, C.c_int64, C.c_int, C.c_double, _vp, _vp]),
    "tg_invert_bases_gf2": (C.c_int, [_vp, _vp, _vp, C.c_int64, C.c_int, _vp]),
    "tg_demo_sample_gf2": (C.c_int, [_vp, _vp, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, _vp, C.c_int64, _vp, _vp, _vp, _vp,
                                     _vp]),
    "tg_expand_f32_gf2": (C.c_int, [_vp, _vp, C.c_int64, C.c_int64, C.c_int, _vp]),
    "tg_demo_gen_gf2": (C.c_int, [C.c_uint64, C.c_uint64, C.c_int64, C.c_int, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_int,
                                  _vp, C.c_int64, _vp, _vp, _vp]),
    "tg_demo_alias_tables_gf2": (C.c_int, [_vp, _vp, C.c_int, C.c_int, _vp]),
    "tg_demo_gen_box": (C.c_int, [C.c_uint64, C.c_uint64, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _vp, _vp,
                                  C.c_int, C.c_int, _vp, C.c_int64, _vp, _vp, _vp]),
    "tg_demo_gen_box_gf2": (C.c_int, [C.c_uint64, C.c_uint64, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _vp,
                                      _vp, C.c_int, C.c_int, _vp, C.c_int64, _vp, _vp, _vp]),
    "tg_change_of_basis_factors": (C.c_int, [_vp, C.c_int64, C.c_int, _vp, C.c_int, _vp, C.c_int64, C.c_int, _vp, C.c_int64,
                                             C.c_int, C.c_int, _vp]),
    "tg_sample_unimodular": (C.c_int, [C.c_uint64, C.c_uint64, C.c_int64, C.c_int, C.c_double, _vp, _vp]),
    "tg_invert_bases": (C.c_int, [_vp, _vp, _vp, C.c_int64, C.c_int, _vp]),
    "tg_mt19937_fill_f64": (C.c_int, [C.c_uint32, C.c_int64, C.c_int64, _vp]),
    "tg_mt19937_fill_f64_state": (C.c_int, [_vp, C.c_int, C.c_int64, C.c_int64, _vp]),
    "tg_demo_from_ustream_workspace": (C.c_int64, [C.c_int64, C.c_int]),
    "tg_demo_from_ustream": (C.c_int, [_vp, C.c_int64, _vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int64, _vp, C.c_int64,
                                       _vp, _vp, _vp, _vp, C.c_int64, _vp]),
    "tg_host_ctx_create": (C.c_int, [C.POINTER(_vp), C.c_int, C.c_int, C.c_int64]),
    "tg_host_ctx_destroy": (C.c_int, [_vp]),
    "tg_step_host": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, C.c_int64, C.c_int]),
    "tg_rollout_host": (C.c_int, [_vp, _vp, _vp, C.c_int, _vp, _vp, _vp, _vp, C.c_int64, C.c_int]),
    "tg_demo_gen_host": (C.c_int, [_vp, C.c_uint64, C.c_uint64, C.c_int64, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_int,
                                   _vp, _vp, _vp]),
    "tg_step_host_i16": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, C.c_int64, C.c_int]),
    "tg_rollout_host_i16": (C.c_int, [_vp, _vp, _vp, C.c_int, _vp, _vp, _vp, _vp, C.c_int64, C.c_int]),
    "tg_step_host_gf2": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, C.c_int64, C.c_int]),
    "tg_rollout_host_gf2": (C.c_int, [_vp, _vp, _vp, C.c_int, _vp, _vp, _vp, _vp, C.c_int64, C.c_int]),
    "tg_demo_gen_host_gf2": (C.c_int, [_vp, C.c_uint64, C.c_uint64, C.c_int64, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_int,
                                       _vp, _vp, _vp]),
}
if TUNING:  # sweep build only (declared under TG_TUNING in include/tensorgame.h)
    _SIGNATURES["tg_tune_step_ctas_per_sm"] = (C.c_int, [C.c_int])
    _SIGNATURES["tg_tune_step_variant"] = (C.c_int, [C.c_int])


def exported_symbols() -> list[str]:
    """Every function include/tensorgame.h declares (used by the symbol test)."""
    import re

    text = HEADER.read_text()
    if not TUNING:  # the sweep-only entry points exist in the -DTG_TUNING build alone
        text = re.sub(r"#ifdef TG_TUNING.*?#endif", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(tg_[a-z0-9_]+)\s*\(", text)))


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if _stale():
            # never load a library built from other sources: the ctypes signatures below describe THIS tree
            try:
                build()
            except (TensorGameError, FileNotFoundError) as e:
                raise TensorGameError(
                    f"{LIB_PATH.name} is missing or older than its sources and could not be rebuilt; "
                    "run `python -c 'import __graft_entry__ as g; g.build()'` (no CPU fallback exists)"
                ) from e
        handle = C.CDLL(str(LIB_PATH))
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        if handle.tg_version() != header_version():
            raise TensorGameError(f"{LIB_PATH.name} reports tg_version {handle.tg_version()}, include/tensorgame.h "
                                  f"declares {header_version()}: rebuild the library")
        _lib = handle
    return _lib


def check(code: int, what: str) -> None:
    if code != TG_OK:
        L = lib()
        msg = L.tg_error_string(code).decode()
        extra = f" (cudaError {L.tg_last_cuda_error()})" if code == -2 else ""
        raise TensorGameError(f"{what}: {msg}{extra}")
