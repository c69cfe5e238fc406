"""Every tensor an env.py wrapper hands to the library is checked for its dtype, exact shape and layout before anything
is launched; the kernels trust every extent, so a wrong-sized buffer must never reach them.

All calls use CPU tensors: a wrong operand fails on its own check, naming it, and a call whose operands are right gets
as far as the device check ("there is no CPU path").  Nothing is launched, so no device is needed.
"""
import ctypes as C

import pytest
import torch

from mat_mul_b200 import env

S, B, R, K = 9, 3, 4, 2
LAY, GW = env.layout(S), env.layout_gf2(S).game_words
GP, TP = LAY.game_pitch, LAY.token_pitch
BOX = (4, 6, 6)


def t(shape, dtype):
    return torch.zeros(shape, dtype=dtype)


def f32(*shape):
    return t(shape, torch.float32)


def i8(*shape):
    return t(shape, torch.int8)


def i16(*shape):
    return t(shape, torch.int16)


def i32(*shape):
    return t(shape, torch.int32)


def i64(*shape):
    return t(shape, torch.int64)


def u8(*shape):
    return t(shape, torch.uint8)


def heads():
    return f32(2 * B, S, S, S)[::2]  # games may sit at any batch stride


def demo_tape(n):
    return u8(R, n + 2, TP)[:, 1:n + 1]  # the steps of a larger store


def _stepper():
    """A HostStepper without a context: its checks need none, and a call that passes them is refused by the library
    for the null context."""
    hs = env.HostStepper.__new__(env.HostStepper)
    hs.S, hs.lay, hs._ctx = S, LAY, C.c_void_p()
    return hs


# (label, call, a maker for each tensor the caller supplies)
NO_CPU = "no CPU path"
CASES = [
    ("pack_states", lambda o: env.pack_states(o["heads"], S, out=o["out"]), dict(heads=heads, out=lambda: i8(B, GP))),
    ("pack_states16", lambda o: env.pack_states16(o["heads"], S), dict(heads=heads)),
    ("expand_states", lambda o: env.expand_states(o["slab"], S, out=o["out"]),
     dict(slab=lambda: i8(B, GP), out=lambda: f32(B + 1, S, S, S)[1:])),
    ("expand_states_bits", lambda o: env.expand_states(o["slab"], S), dict(slab=lambda: i32(B, GW))),
    ("expand_states16", lambda o: env.expand_states16(o["slab16"], S, out=o["out"]),
     dict(slab16=lambda: i16(B, GP), out=lambda: f32(B, S, S, S))),
    ("pack_actions", lambda o: env.pack_actions(o["actions"], S), dict(actions=lambda: i64(B, 3 * S))),
    ("unpack_actions", lambda o: env.unpack_actions(o["tape"], S), dict(tape=lambda: u8(B, TP))),
    ("pack_gf2", lambda o: env.pack_gf2(o["slab"], S), dict(slab=lambda: i16(B, GP))),
    ("unpack_gf2", lambda o: env.unpack_gf2(o["bits"], S), dict(bits=lambda: i32(B, GW))),
    ("step_batch", lambda o: env.step_batch(o["slab"], o["tape"], S, 1, out=o["out"], flags=o["flags"], nnz=o["nnz"]),
     dict(slab=lambda: i8(B, GP), tape=lambda: u8(B, TP), out=lambda: i8(B, GP), flags=lambda: u8(B), nnz=lambda: i32(B))),
    ("step_batch_i16", lambda o: env.step_batch(o["slab"], o["tape"], S, 1, out=o["out"]),
     dict(slab=lambda: i16(B, GP), tape=lambda: u8(B, TP), out=lambda: i16(B, GP))),
    ("step_batch_bits", lambda o: env.step_batch(o["slab"], o["tape"], S, 1, out=o["out"]),
     dict(slab=lambda: i32(B, GW), tape=lambda: u8(B, TP), out=lambda: i32(B, GW))),
    ("expand_children", lambda o: env.expand_children(o["slab"], o["tape"], S, 1),
     dict(slab=lambda: i8(B, GP), tape=lambda: u8(B, 5, TP))),
    ("rollout", lambda o: env.rollout(o["slab"], o["tape"], S, 1, out=o["out"]),
     dict(slab=lambda: i16(B, GP), tape=lambda: u8(K, B, TP), out=lambda: i16(B, GP))),
    ("replay", lambda o: env.replay(o["slab"], o["tape"], S, 1, out=o["out"]),
     dict(slab=lambda: i32(B, GW), tape=lambda: u8(K, B, TP), out=lambda: i32(B, GW))),
    ("make_synthetic_demos", lambda o: env.make_synthetic_demos(B, R, S, device="cpu", tape=o["tape"], slab=o["slab"]),
     dict(tape=lambda: demo_tape(B), slab=lambda: i8(B + 2, GP)[1:B + 1])),
    ("make_synthetic_demos_gf2", lambda o: env.make_synthetic_demos_gf2(B, R, S, device="cpu", tape=o["tape"], bits=o["bits"]),
     dict(tape=lambda: demo_tape(B), bits=lambda: i32(B, GW))),
    ("make_synthetic_demos_box", lambda o: env.make_synthetic_demos_box(B, R, S, BOX, device="cpu", tape=o["tape"],
                                                                         slab=o["slab"]),
     dict(tape=lambda: demo_tape(B), slab=lambda: i8(B, GP))),
    ("make_synthetic_demos_box_gf2", lambda o: env.make_synthetic_demos_box_gf2(B, R, S, BOX, device="cpu", tape=o["tape"],
                                                                                 bits=o["bits"]),
     dict(tape=lambda: demo_tape(B), bits=lambda: i32(B, GW))),
    ("accumulate_demos", lambda o: env.accumulate_demos(o["tape"], S, 1, slab=o["slab"]),
     dict(tape=lambda: u8(R, B, TP), slab=lambda: i8(B, GP))),
    ("accumulate_demos16", lambda o: env.accumulate_demos16(o["tape"], S, 1, slab16=o["slab16"]),
     dict(tape=lambda: u8(R, B, TP), slab16=lambda: i16(B, GP))),
    ("accumulate_demos_tc", lambda o: env.accumulate_demos_tc(o["tape"], 1, slab=o["slab"]),
     dict(tape=lambda: u8(R, B, 48), slab=lambda: i8(B, 4096))),
    ("demo_samples", lambda o: env.demo_samples(o["tape"], o["slab"], o["idx"], S, 2),
     dict(tape=lambda: u8(R, B, TP), slab=lambda: i8(B, GP), idx=lambda: i64(7))),
    ("DemoStore", lambda o: env.DemoStore(o["records"], o["targets"], S, 1),
     dict(records=lambda: u8(B, R, TP), targets=lambda: i16(B, GP))),
    ("DemoStore_bits", lambda o: env.DemoStore(o["records"], o["targets"], S, 1),
     dict(records=lambda: u8(B, R, TP), targets=lambda: i32(B, GW))),
    ("DemoStore.from_tape", lambda o: env.DemoStore.from_tape(o["tape"], i8(B, GP), S, 1), dict(tape=lambda: u8(R, B, TP))),
    ("slice_rank", lambda o: env.slice_rank(o["slab"], S), dict(slab=lambda: i8(B, GP))),
    ("state_keys", lambda o: env.state_keys(o["slab"], S), dict(slab=lambda: i16(B, GP))),
    ("change_of_basis", lambda o: env.change_of_basis(o["slab"], o["mats"], S, tape=o["tape"], out=o["out"]),
     dict(slab=lambda: i8(B, GP), mats=lambda: i8(B, 3, S, S), tape=lambda: u8(R, B, TP), out=lambda: i16(B, GP))),
    ("change_of_basis_factors", lambda o: env.change_of_basis_factors(o["tape"], o["mats"], S, 1),
     dict(tape=lambda: u8(R, B, TP), mats=lambda: i8(3, S, S))),
    ("invert_bases", lambda o: env.invert_bases(o["mats"], out=o["out"]),
     dict(mats=lambda: i8(B, 3, S, S), out=lambda: i8(B, 3, S, S))),
    ("change_of_basis_gf2", lambda o: env.change_of_basis_gf2(o["bits"], o["mats"], S, tape=o["tape"], out=o["out"]),
     dict(bits=lambda: i32(B, GW), mats=lambda: i32(1, 3, S), tape=lambda: u8(R, B, TP), out=lambda: i32(B, GW))),
    ("change_of_basis_factors_gf2", lambda o: env.change_of_basis_factors_gf2(o["tape"], o["mats"], S),
     dict(tape=lambda: u8(R, B, TP), mats=lambda: i32(B, 3, S))),
    ("invert_bases_gf2", lambda o: env.invert_bases_gf2(o["mats"], out=o["out"]),
     dict(mats=lambda: i32(B, 3, S), out=lambda: i32(B, 3, S))),
    ("HostStepper.step", lambda o: _stepper().step(o["slab"], o["tape"], o["out"], o["flags"], o["nnz"], 1),
     dict(slab=lambda: i8(B, GP), tape=lambda: u8(B, TP), out=lambda: i8(B, GP), flags=lambda: u8(B), nnz=lambda: i32(B))),
    ("HostStepper.step_i16", lambda o: _stepper().step(o["slab"], o["tape"], o["out"], o["flags"], o["nnz"], 1),
     dict(slab=lambda: i16(B, GP), tape=lambda: u8(B, TP), out=lambda: i16(B, GP), flags=lambda: u8(B), nnz=lambda: i32(B))),
    ("HostStepper.rollout", lambda o: _stepper().rollout(o["slab"], o["tape"], o["out"], o["flags"], o["nnz"], o["steps"], 1),
     dict(slab=lambda: i8(B, GP), tape=lambda: u8(K, B, TP), out=lambda: i8(B, GP), flags=lambda: u8(B), nnz=lambda: i32(B),
          steps=lambda: i32(B))),
    ("HostStepper.rollout_bits", lambda o: _stepper().rollout(o["slab"], o["tape"], o["out"], o["flags"], o["nnz"], o["steps"], 1),
     dict(slab=lambda: i32(B, GW), tape=lambda: u8(K, B, TP), out=lambda: i32(B, GW), flags=lambda: u8(B), nnz=lambda: i32(B),
          steps=lambda: i32(B))),
    ("HostStepper.make_demos", lambda o: _stepper().make_demos(o["tape"], o["slab"], o["flags"], 1, (-1, 0, 1), (0.2, 0.6, 0.2)),
     dict(tape=lambda: u8(R, B, TP), slab=lambda: i8(B, GP), flags=lambda: u8(B))),
    ("HostStepper.make_demos_bits", lambda o: _stepper().make_demos(o["tape"], o["slab"], o["flags"], 1, (-1, 0, 1),
                                                                    (0.2, 0.6, 0.2)),
     dict(tape=lambda: u8(R, B, TP), slab=lambda: i32(B, GW), flags=lambda: u8(B))),
]
ANY_LAYOUT = {("DemoStore", "targets"), ("DemoStore_bits", "targets")}  # copied to a contiguous store
ANY_SHAPE = {("demo_samples", "idx"),  # any shape of nb indices
             ("invert_bases_gf2", "mats")}  # (N, 3, S): the matrices set the call's N and S


def _ok(label):
    return "bad argument" if label.startswith("HostStepper") else NO_CPU


def _short(x):
    """x one element short along its last dimension (one row short for a vector)."""
    return x[..., :-1].contiguous()


def _strided(x):
    """A non-contiguous view of x's shape, dtype and values."""
    return torch.stack((x, x), dim=-1)[..., 0]


def _wrong_operands():
    for kind, exempt in (("dtype", set()), ("short", ANY_SHAPE), ("strided", ANY_LAYOUT)):
        for label, call, ops in CASES:
            for name in ops:
                if (label, name) not in exempt:
                    yield pytest.param(kind, call, ops, name, id=f"{label}-{name}-{kind}")


@pytest.mark.parametrize("label, call, ops", [pytest.param(*c, id=c[0]) for c in CASES])
def test_correct_operands_reach_the_device_check(label, call, ops):
    with pytest.raises(env.TensorGameError, match=_ok(label)):
        call({k: make() for k, make in ops.items()})


@pytest.mark.parametrize("kind, call, ops, name", list(_wrong_operands()))
def test_wrong_operand_is_refused_by_name(kind, call, ops, name):
    o = {k: make() for k, make in ops.items()}
    x = o[name]
    o[name] = {"dtype": lambda: x.to(torch.float64), "short": lambda: _short(x), "strided": lambda: _strided(x)}[kind]()
    with pytest.raises(env.TensorGameError, match=rf"^{name} "):
        call(o)


def test_int16_targets_are_refused_by_make_demos():
    with pytest.raises(env.TensorGameError, match="not int16 targets"):
        _stepper().make_demos(u8(R, B, TP), i16(B, GP), u8(B), 1, (-1, 0, 1), (0.2, 0.6, 0.2))
