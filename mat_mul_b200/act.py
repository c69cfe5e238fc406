"""Drop-in for the reference's act.py (/root/reference/act.py): same function
names, signatures and return values.  The environment work of the search --
child expansion, null-action pruning, terminal test, tree keys, rank reward --
runs in the sm_100a kernels (tg_step, tg_state_key, tg_slice_rank); the search
bookkeeping itself stays host-side Python as in the reference (it is
model-bound: SURVEY.md 3.2).

Tree keys are the kernel's 64-bit state keys (ints) instead of the reference's
"_".join strings (utils.py:164-169); mc_tree / state_info keep the reference's
layout otherwise: state_info[key] = (candidate_states, 0, 0, visit_count,
q_values, actions), mc_tree[key] = [child keys].

Star-import surface: Dict, List, torch, AlphaTensor (when the reference's
model.py is importable) and everything from utils.
"""
from typing import Dict, List

import torch

try:  # the reference's network; out of scope and consumed unchanged (model.py)
    from model import AlphaTensor
except ImportError:  # pragma: no cover - model.py is not part of this package
    AlphaTensor = None

from mat_mul_b200 import env as _env
from mat_mul_b200.utils import *  # noqa: F401,F403
from mat_mul_b200.utils import _COEF_SHIFT, ChildStates, _device, _heads_to_slab, _slab_to_heads

_MAX_EXPANSION_TRIES = 1000  # the reference loops forever when every sampled child is null or known (SURVEY Q11)


def _head_key(state: torch.Tensor) -> int:
    """Tree key of a (1, T, S, S, S) state: tg_state_key of its head."""
    S = state.shape[-1]
    return int(_env.state_keys(_heads_to_slab(state[:, 0], S), S)[0].item())


def get_child_states(state: torch.Tensor, actions: torch.Tensor, vec_cardinality=5):
    """act.py:266-275: for each of the k sampled actions, new_head = head - action_to_tensor(action) (token shift
    fixed at 1) and history = the previous slots shifted by one.  One tg_expand_children launch; the returned
    list also carries the kernel's per-child flags (ChildStates)."""
    bs, k = actions.shape[:2]
    S = state.shape[-1]
    dev = _device()
    head = _heads_to_slab(state[:, 0], S)                                   # (bs, GP), int8 or int16
    # the reference's coefficient is token - 1 whatever the alphabet (action_to_tensor, SURVEY Q1): re-based to the
    # kernels' widest alphabet (token + 3, shift 4) so that the token bound of the packed arithmetic holds
    tape = _env.pack_actions(actions.reshape(bs * k, -1).to(dev).to(torch.int64).contiguous(), S,
                             rebase=_COEF_SHIFT - 1).reshape(bs, k, -1)
    # one launch: the k children of every state, their null / terminal flags, non-zero counts and state keys (K8)
    out, flags, nnz, keys = _env.expand_children(head, tape, S, _COEF_SHIFT)
    if head.dtype == torch.int8 and bool((flags & _env.FLAG_RANGE).any()):
        # the reference computes in float32 and never wraps: children the int8 slab cannot hold are made from the int16
        # slab of the same values (same element layout)
        out, flags, nnz, keys = _env.expand_children(head.to(torch.int16), tape, S, _COEF_SHIFT)
    if bool((flags & _env.FLAG_RANGE).any()):
        raise _env.TensorGameError("get_child_states: a child state left the int16 slab's guaranteed range [-16384, 16383]")
    new_heads = _slab_to_heads(out.reshape(bs * k, -1), S, (bs, k), state.dtype, state.device)
    children = ChildStates(torch.cat([new_heads[:, i : i + 1], state[:, :-1]], dim=1) for i in range(k))
    f = flags.reshape(bs, k)
    children.parent = state
    children.range_flags = ((f & _env.FLAG_RANGE) != 0).any(0).cpu()
    children.null_flags = ((f & _env.FLAG_NULL) != 0).all(0).cpu()
    children.terminal = ((f & _env.FLAG_TERMINAL) != 0).all(0).cpu()
    children.nnz = nnz.reshape(bs, k).cpu()
    children.keys = keys.reshape(bs, k)[0].cpu()
    return children


def select_next_state(candidate_states: List[torch.Tensor], q_vals: torch.Tensor, visit_count: torch.Tensor,
                      reps: Dict[int, list], c1=1.25, c2=19652.0, return_idx: bool = False):
    """act.py:240-263: UCB argmax.  (pi counts repetitions, which the callers always pass empty.)"""
    pi = torch.tensor([len(reps[i]) for i in range(len(candidate_states)) if i in reps]).to(q_vals.device)
    if pi.shape[0] != visit_count.shape[1]:
        pi = pi[: visit_count.shape[1]]
    total = visit_count.sum()
    explore = c1 + torch.log((total + c2 + 1) / c2)
    ucb = q_vals.reshape(-1) + explore * pi * torch.sqrt(total) / (1 + visit_count)
    best = ucb.argmax()
    return best if return_idx else candidate_states[best]


def backward_pass(trajectory, state_info, leaf_q_val):
    """act.py:219-237: propagate the leaf value up the trajectory, -1 per edge, running-mean Q."""
    new_state_info = state_info.copy()
    reward = 0
    for key, action_idx in reversed(trajectory):
        if action_idx is None:
            reward += leaf_q_val
            continue
        _, _, _, visits, q, _ = new_state_info[key]
        if isinstance(reward, torch.Tensor):
            reward = reward.to(q.device)
        a = int(action_idx)
        reward -= 1
        q[:, a] = (visits[:, a] * q[:, a] + reward) / (visits[:, a] + 1)
        visits[:, a] += 1
    return new_state_info


@torch.no_grad()
def extend_tree(model, state: torch.Tensor, i_action: int, max_actions: int, mc_tree: Dict, state_info: Dict, horizon=5):
    """act.py:115-216: walk the tree from `state` by UCB to an unexpanded node, expand it with the model's sampled
    actions (children through get_child_states; null and already-known children pruned) and back the value up."""
    new_state_info = state_info.copy()
    new_mc_tree = mc_tree.copy()
    idx = i_action
    max_actions_mc = min(max_actions, i_action + horizon)
    key = _head_key(state)
    trajectory = []
    while key in new_mc_tree:
        candidates, _, _, visits, q, _ = new_state_info[key]
        pick = select_next_state(candidates, q, visits, {i: [] for i in range(len(candidates))}, return_idx=True)
        trajectory.append((key, pick))
        if len(trajectory) > 2 * max_actions:
            print("trajectory too long")
        state = candidates[pick]
        key = new_mc_tree[trajectory[-1][0]][int(pick)]  # child keys were stored when the node was expanded
        idx += 1
    if idx <= max_actions_mc:
        trajectory.append((key, None))
        if tensor_factorized(get_head_state(state)):
            # the reference leaves leaf_q_val unassigned on this path and fails in backward_pass (act.py:177-215)
            raise UnboundLocalError("cannot access local variable 'leaf_q_val' where it is not associated with a value")
        state = state.to(model.device)
        scalars = get_scalars(state, idx).to(model.device)
        candidates, cand_keys, tries = [], [], 0
        while len(candidates) == 0:
            tries += 1
            if tries > _MAX_EXPANSION_TRIES:
                raise RuntimeError("extend_tree: the model keeps proposing null or already-expanded children")
            actions, _, q_vals = model.fwd_infer(state, scalars)
            children = get_child_states(state, actions)
            keep = remove_null_actions(state, children)
            child_keys = children.keys.tolist()
            keep = [i for i in keep if child_keys[i] not in new_mc_tree]
            actions = actions[:, keep]
            candidates = [children[i] for i in keep]
            cand_keys = [child_keys[i] for i in keep]
        kept_actions = actions.to("cpu")
        kept_q = torch.zeros(kept_actions.shape[:-1])
        new_state_info[key] = (candidates, 0, 0, torch.zeros_like(kept_q), kept_q, kept_actions)
        new_mc_tree[key] = cand_keys
        leaf_q_val = q_vals
    else:
        leaf_q_val = -get_rank(state)
    new_state_info = backward_pass(trajectory, new_state_info, leaf_q_val)
    return new_mc_tree, new_state_info


def mc_ts(model, root_state: torch.Tensor, n_sim: int, i_action: int, max_actions: int, mc_tree: dict, state_info: dict):
    """act.py:67-112: n_sim tree extensions from the root (minus the visits it already has), then the child with
    the best Q is played."""
    key = _head_key(root_state)
    if key in state_info:
        with torch.no_grad():
            n_sim = max(n_sim - int(state_info[key][3].sum()), 0)
    for _ in range(n_sim):
        mc_tree, state_info = extend_tree(model, root_state, i_action, max_actions, mc_tree, state_info)
    candidates, _, _, visits, q, _ = state_info[key]
    pick = select_next_state(candidates, q, visits, {i: [] for i in range(len(candidates))}, return_idx=True)
    return candidates[pick], mc_tree, state_info


@torch.no_grad()
def get_improved_policy(state_info: Dict, string_seq: List, n_steps: int, n_logits: int, n_bar: int):
    """act.py:278-301: visit counts tempered by tau = log(N)/log(n_bar) when N > n_bar, spread over the tokens of
    each sampled action -> (len(seq), n_steps, n_logits)."""
    policy_seq = torch.zeros(len(string_seq), n_steps, n_logits)
    n_bar = torch.tensor(n_bar)
    steps = torch.arange(n_steps)
    for ii, key in enumerate(string_seq):
        _, _, _, visits, _, action_cands = state_info[key]
        total = visits.sum()
        tau = (total.log() / n_bar.log()).item() if total > n_bar else 1
        improved = visits ** (1 / tau) / total
        for sample_id in range(action_cands.shape[1]):
            tokens = action_cands[0, sample_id]
            policy_seq[ii, steps[: len(tokens)], tokens] += improved[0, sample_id]
    return policy_seq


def actor_prediction(model, initial_state: torch.Tensor, max_actions: int, n_sim: int, n_bar: int):
    """act.py:8-64: one game by MCTS -> (state_seq, policy_seq, reward_seq); reward_seq is the cumulative sum of
    -1 per action with -get_rank(final state) added to the last one."""
    state = initial_state.unsqueeze(0)
    state_seq, key_seq = [], []
    mc_tree, state_info = {}, {}
    i_action = 0
    while i_action < max_actions:
        state_seq.append(state)
        key_seq.append(_head_key(state))
        state, mc_tree, state_info = mc_ts(model, state, n_sim, i_action, max_actions, mc_tree, state_info)
        if tensor_factorized(state):  # sees all dim_t slots of the batched state (SURVEY Q3)
            break
        i_action += 1
    policy_seq = get_improved_policy(state_info, key_seq, model.n_steps, model.n_logits, n_bar)
    end_state_reward = -get_rank(state)
    reward_seq = torch.cumsum(torch.tensor([-1] * (len(policy_seq) - 1) + [-1 + end_state_reward]), dim=0)
    return [s.squeeze(0) for s in state_seq], policy_seq, reward_seq
