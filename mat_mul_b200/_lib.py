"""Loader for libtensorgame_b200.so (the C-ABI CUDA library, include/tensorgame.h).

The library is built in-tree with nvcc for sm_100a only.  There is no CPU
fallback: if the library cannot be loaded, every compute entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os
import re
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

# ctypes of the header's scalar types; pointers are mapped in _ctype
_SCALARS = {"int": C.c_int, "int64_t": C.c_int64, "uint64_t": C.c_uint64, "uint32_t": C.c_uint32, "double": C.c_double}


def _ctype(decl: str, ret: bool = False):
    """The ctypes type of a C type as include/tensorgame.h writes it (a return type, or a parameter without its name).
    Raises for a type it does not know: a guessed type would pass wrong arguments without any error."""
    words = [w for w in decl.replace("*", " * ").split() if w != "const"]
    stars, base = words.count("*"), " ".join(w for w in words if w != "*")
    if not stars and base in _SCALARS:
        return _SCALARS[base]
    if (base, stars) == ("char", 1) and ret:
        return C.c_char_p
    if (base, stars) == ("int", 1):
        return C.POINTER(C.c_int)
    if (base, stars) == ("tg_host_ctx", 2):
        return C.POINTER(C.c_void_p)
    if stars and not ret:
        return C.c_void_p
    raise TensorGameError(f"{HEADER.name}: no ctypes type for {decl.strip()!r}")


def _parse_prototypes(text: str) -> dict:
    """name -> (restype, argtypes) of every tg_* function a C header declares; the TG_TUNING block counts only in the
    sweep build, as there the library exports it."""
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    if not TUNING:
        text = re.sub(r"#ifdef TG_TUNING.*?#endif", "", text, flags=re.S)
    text = re.sub(r"^\s*#.*$", "", text, flags=re.M)
    sigs = {}
    for ret, name, params in re.findall(r"([^;{}()]*?)\b(tg_\w+)\s*\(([^()]*)\)\s*;", text):
        params = [p.strip() for p in params.split(",")]
        if params == ["void"]:
            params = []
        # every parameter is named in the header: the type is what precedes the name
        sigs[name] = (_ctype(ret, ret=True), [_ctype(re.fullmatch(r"(.*?)\w+", p, flags=re.S).group(1)) for p in params])
    return sigs


_SIGNATURES = _parse_prototypes(HEADER.read_text())


def exported_symbols() -> list[str]:
    """Every function include/tensorgame.h declares (used by the symbol test)."""
    return sorted(_SIGNATURES)


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if _stale():
            # never load a library built from other sources: the ctypes signatures come from THIS tree's header
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
