"""Drop-in for the reference's utils.py (same names, signatures, dtypes, shapes
and quirks; /root/reference/utils.py).  Every tensor-game computation runs in
the sm_100a kernels behind include/tensorgame.h; there is no CPU arithmetic
path -- inputs living on the CPU are moved to the CUDA device, processed there
and the result is returned on the caller's device, as the reference would.

Star-import surface (the reference has no __all__): torch, Categorical, List,
Tuple and every function below.  Sizes: dim_3d in {4, 9, 16, 25}; factor
coefficients in [-4, 4] (the game's alphabet is {-2..2}).
"""
from typing import List, Tuple  # noqa: F401  (part of the reference's star-import surface)

import os

import torch
from torch.distributions.categorical import Categorical  # noqa: F401

from mat_mul_b200 import env as _env
from mat_mul_b200._lib import TensorGameError

_COEF_SHIFT = 4  # internal token shift when a caller hands raw coefficients


def _device() -> torch.device:
    if not torch.cuda.is_available():
        raise TensorGameError("mat_mul_b200 needs a CUDA device (B200); there is no CPU fallback")
    return torch.device("cuda", int(os.environ.get("TG_DEVICE", torch.cuda.current_device())))


def _heads_to_slab(heads: torch.Tensor, S: int) -> torch.Tensor:
    """(..., S, S, S) tensor of any dtype/device -> slab (N, GP) on the CUDA device: int8 whenever every value is an
    integer in [-128, 127], int16 otherwise (the reference computes in float32 and has no such limit).  Raises if a
    value is not an integer in [-32768, 32767].  The one place the mirrors choose a slab format."""
    h = heads.reshape(-1, S, S, S).to(device=_device(), dtype=torch.float32).contiguous()
    try:
        return _env.pack_states(h, S)
    except TensorGameError:
        return _env.pack_states16(h, S)


def _slab_to_heads(slab: torch.Tensor, S: int, shape, dtype, device) -> torch.Tensor:
    out = _env.expand_states16(slab, S) if slab.dtype == torch.int16 else _env.expand_states(slab, S)
    return out.reshape(*shape, S, S, S).to(device=device, dtype=dtype)


class ChildStates(list):
    """The list get_child_states returns, carrying what the step kernel already knows about every child."""

    parent = None       # the state tensor the children were expanded from
    range_flags = None  # bool (k,): the child left the guaranteed zone of the slab it was computed in (always False: a
    #                     child that leaves the int8 zone is recomputed on an int16 slab, and leaving the int16 zone raises)
    null_flags = None   # bool (k,): child head == parent head (utils.py:191-194)
    terminal = None     # bool (k,): child head all zero
    nnz = None          # int32 (k,)
    keys = None         # int64 (k,): tg_state_key of the child heads


# ------------------------------------------------------------------ glue (no tensor-game arithmetic)
def print_params(model):
    """utils.py:7-19"""
    total = sum(p.numel() for p in model.parameters())
    pol = sum(p.numel() for p in model.policy_head.parameters())
    print(f"{total // int(1e6)}M parameters")
    print(f"{total // int(1e3)}k parameters")
    print(f"{sum(p.numel() for p in model.torso.parameters())} parameters: torso")
    print(f"{pol // int(1e6)}M parameters: policy head")
    print(f"{pol} parameters: policy head")
    print(f"{sum(p.numel() for p in model.value_head.parameters())} parameters: value head")


def get_scalars(tt: torch.Tensor, t_step: int, batch_size=True):
    """utils.py:22-37: (B, 1) float32 filled with t_step, or a (1,) tensor for a single example."""
    if batch_size:
        return torch.full((tt.shape[0], 1), float(t_step))
    return torch.tensor(t_step).unsqueeze(0).float()


def action_to_uvw(action: torch.Tensor, shift=1):
    """utils.py:56-66: (*, 3S) tokens -> three (*, S) coefficient tensors (token - shift)."""
    dim_3d = action.shape[-1] // 3
    return (action - shift).split(dim_3d, dim=-1)


def get_head_state(state: torch.Tensor, unsqueeze=True):
    """utils.py:99-111"""
    head = state[:, 0]
    return head.unsqueeze(1) if unsqueeze else head


def state_to_str(state: torch.Tensor):
    """utils.py:164-169 (the batched path uses tg_state_key instead, see act.py)."""
    return "_".join(str(v) for v in state.reshape(-1).long().detach().cpu().tolist())


def str_to_state(string: str, shape: tuple) -> torch.Tensor:
    """utils.py:172-178"""
    return torch.tensor([float(x) for x in string.split("_")]).reshape(shape)


def factor_sample(values, probs, dim_3d):
    """utils.py:197-200.  One Categorical draw of dim_3d entries from torch's generator; batched
    generation goes through create_synthetic_demo / SyntheticDemoDataset (tg_demo_from_ustream)."""
    return values[Categorical(probs).sample(torch.Size([dim_3d]))]


def build_matmul_tensor(dim_t: int, dim_i: int, dim_j: int, dim_k: int):
    """utils.py:143-161: slot 0 holds the matmul tensor, T[0, (ik//J)*K + j, j*J + ik%J, ik] = 1; built once on
    the host like the reference (valid for square sizes only, SURVEY Q8: other shapes raise IndexError)."""
    out = torch.zeros(dim_t, dim_i * dim_j, dim_j * dim_k, dim_i * dim_k)
    ik = torch.arange(dim_i * dim_k).repeat_interleave(dim_j)
    j = torch.arange(dim_j).repeat(dim_i * dim_k)
    rows, cols = (ik // dim_j) * dim_k + j, j * dim_j + ik % dim_j
    if int(rows.max()) >= out.shape[1] or int(cols.max()) >= out.shape[2]:
        raise IndexError("build_matmul_tensor: index out of range (the reference only supports square sizes)")
    out[0, rows, cols, ik] = 1
    return out


def update_state(state: torch.Tensor, action: torch.Tensor, batch=True):
    """utils.py:114-131 -- dead code in the reference (never called; ADDS the action and mis-slices when
    batch=False, SURVEY Q5).  Kept importable with the same behaviour."""
    if batch:
        head = (state[:, 0] + action_to_tensor(action.squeeze())).unsqueeze(1)
        return torch.cat((head, state[:, :-1]), dim=1)
    head = get_head_state(state) + action_to_tensor(action)
    return torch.cat((head, state[:-1]), dim=0)


# ------------------------------------------------------------------ kernels
def uvw_to_tensor(uvw: Tuple[torch.Tensor, torch.Tensor, torch.Tensor]):
    """utils.py:69-85: rank-1 tensor u_i v_j w_k for (*, S) factors -> (*, S, S, S), dtype of the inputs.
    Runs tg_demo_accumulate with R = 1."""
    uu, vv, ww = uvw
    S = uu.shape[-1]
    lead = uu.shape[:-1]
    coef = torch.cat((uu.reshape(-1, S), vv.reshape(-1, S), ww.reshape(-1, S)), dim=1)
    if coef.numel() and int(coef.abs().max()) > _COEF_SHIFT:
        raise TensorGameError(f"factor coefficients must be in [-{_COEF_SHIFT}, {_COEF_SHIFT}]")
    tokens = (coef.to(torch.int64) + _COEF_SHIFT).to(_device())
    tape = _env.pack_actions(tokens, S).unsqueeze(0)
    slab, _ = _env.accumulate_demos(tape, S, _COEF_SHIFT)
    return _slab_to_heads(slab, S, lead, uu.dtype, uu.device)


def action_to_tensor(action: torch.Tensor):
    """utils.py:88-96: rank-1 tensor of an action; the token shift is FIXED at 1 here (SURVEY Q1)."""
    return uvw_to_tensor(action_to_uvw(action))


def uvw_to_demo(uu: torch.Tensor, vv: torch.Tensor, ww: torch.Tensor, device: str, shift=1):
    """utils.py:40-53: (sum of the n rank-1 terms as a float32 (4,4,4) tensor, tokens cat(u,v,w)+shift).
    The reference hard-codes 4x4x4 (SURVEY Q7)."""
    if uu.shape[-1] != 4:
        raise RuntimeError("uvw_to_demo: the reference accumulates into a hard-coded (4, 4, 4) tensor")
    action_list = torch.cat((uu, vv, ww), dim=1)
    action_list += shift
    tokens = (action_list.to(torch.int64) - shift + _COEF_SHIFT).to(_device())
    tape = _env.pack_actions(tokens, 4).unsqueeze(1)  # (R, 1, TP): one demo of R steps
    slab, _ = _env.accumulate_demos(tape, 4, _COEF_SHIFT)
    mult_tensor = _env.expand_states(slab, 4)[0].to(device)
    return mult_tensor, action_list


def get_rank(state: torch.Tensor):
    """utils.py:134-140: int(sum over batch and slices T[i,:,:] of the matrix rank) -- tg_slice_rank (exact)."""
    head = get_head_state(state, unsqueeze=False)
    S = head.shape[-1]
    return int(_env.slice_rank(_heads_to_slab(head, S), S).sum().item())


def tensor_factorized(state):
    """utils.py:181-188: (state[0] == 0).all() -- note it indexes dim 0, so a batched (1,T,S,S,S) state tests ALL
    T slots (SURVEY Q3).  Every (S,S,S) block of state[0] goes through the kernel's all-zero flag."""
    x = state[0]
    S = x.shape[-1]
    if x.dim() < 3 or x.shape[-3:] != (S, S, S):
        raise TensorGameError("tensor_factorized expects (..., S, S, S) blocks")
    slab = _heads_to_slab(x, S)
    empty_tape = torch.empty((0, slab.shape[0], _env.layout(S).token_pitch), dtype=torch.uint8, device=slab.device)
    _, flags, _, _ = _env.rollout(slab, empty_tape, S, 1)
    return ((flags & _env.FLAG_TERMINAL) != 0).all().to(state.device)


def remove_null_actions(state: torch.Tensor, candidate_states: List[torch.Tensor]):
    """utils.py:191-194: indexes of candidates whose head differs from the state's head.  Children made by
    get_child_states already carry the kernel's NULL flag; other lists are compared on the device."""
    if isinstance(candidate_states, ChildStates) and candidate_states.parent is state:
        return [i for i, null in enumerate(candidate_states.null_flags.tolist()) if not null]
    S = state.shape[-1]
    ref = _heads_to_slab(state[:, 0], S)
    idxs = []
    for i, c in enumerate(candidate_states):
        if bool((_heads_to_slab(c[:, 0], S) != ref).any()):
            idxs.append(i)
    return idxs


def create_synthetic_demo(values: Tuple[int], probs: Tuple[int], n_actions: int, dim_3d: int, shift: int):
    """utils.py:203-233: (list of n_actions (3S,) int64 token tensors, float32 (S,S,S) target), drawn from
    torch's global CPU generator exactly as the reference's rejection loop does (tg_demo_from_ustream);
    the generator is left where the reference would leave it."""
    vals = [int(v) for v in torch.as_tensor(values).tolist()]
    pr = [float(p) for p in torch.as_tensor(probs).tolist()]
    tape, slab, _, _ = _env.demos_from_seed(1, n_actions, dim_3d, vals, pr, shift, seed=None, device=_device())
    tokens = _env.unpack_actions(tape.reshape(n_actions, -1), dim_3d).cpu()
    action_seq = [tokens[r] for r in range(n_actions)]
    target_tensor = _env.expand_states(slab, dim_3d)[0].cpu()
    return action_seq, target_tensor
