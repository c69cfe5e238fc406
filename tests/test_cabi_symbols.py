"""CPU-side checks of the drop-in boundary: the C-ABI library loads, exports every
symbol include/tensorgame.h declares, and refuses to compute without a GPU."""
import ctypes as C

import pytest

from mat_mul_b200 import _lib


def test_library_exports_every_declared_symbol():
    L = _lib.lib()
    names = _lib.exported_symbols()
    assert "tg_step" in names and "tg_layout" in names and len(names) >= 10
    for name in names:
        assert hasattr(L, name), f"{name} declared in tensorgame.h but not exported"
    assert L.tg_version() == _lib.header_version() >= 200


def test_layout_contract():
    L = _lib.lib()
    rp, gp, tp = C.c_int(), C.c_int(), C.c_int()
    want = {4: (16, 64, 16), 9: (84, 768, 32), 16: (256, 4096, 48)}
    for S, w in want.items():
        assert L.tg_layout(S, C.byref(rp), C.byref(gp), C.byref(tp)) == 0
        assert (rp.value, gp.value, tp.value) == w
    assert L.tg_layout(5, None, None, None) == -1  # TG_E_ARG
    assert L.tg_error_string(-1) == b"bad argument"


def test_no_cpu_fallback():
    import torch

    from mat_mul_b200 import env

    slab = torch.zeros((2, 768), dtype=torch.int8)
    tape = torch.zeros((2, 32), dtype=torch.uint8)
    with pytest.raises(env.TensorGameError):
        env.step_batch(slab, tape, 9, 2)


def test_host_mt19937_stream_matches_torch():
    # host-side logic of parity-mode demo generation: the library's MT19937 continues torch's CPU generator
    import numpy as np
    import torch

    from mat_mul_b200 import env

    torch.manual_seed(5)
    a = env.torch_cpu_stream(10)
    assert np.array_equal(a, torch.rand(10, dtype=torch.float64).numpy())
    c = env.torch_cpu_stream(700)  # crosses a twist, starts mid-state
    assert np.array_equal(c, torch.rand(700, dtype=torch.float64).numpy())
    assert np.array_equal(env.torch_cpu_stream(5, seed=5), a[:5])
    assert np.array_equal(env.torch_cpu_stream(5, seed=5, skip=3), a[3:8])
    g = torch.Generator().manual_seed(77)
    x = env.torch_cpu_stream(1300, generator=g)
    assert np.array_equal(x, torch.rand(1300, dtype=torch.float64, generator=g).numpy())
