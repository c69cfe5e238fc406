"""Drop-in for the reference's datasets.py (/root/reference/datasets.py): same
class names, constructor arguments, item shapes/dtypes and constants.  Demo
generation and per-sample reconstruction run in the sm_100a kernels
(tg_demo_from_ustream, tg_demo_accumulate, tg_demo_sample); the demo store
lives in HBM instead of two .pt files per demo, with one consolidated file in
save_dir for the reference's overwrite/resume semantics (datasets.py:48-72).

Star-import surface: np, Path, List, torch, Categorical, Dataset, everything
from utils, the SAVE_DIR_* / *_BUFFER_SIZE constants and the classes below.
"""
import numpy as np
from pathlib import Path
from typing import List

import torch
from torch.distributions.categorical import Categorical
from torch.utils.data import Dataset

from mat_mul_b200 import env as _env
from mat_mul_b200.utils import *  # noqa: F401,F403
from mat_mul_b200.utils import _device, _COEF_SHIFT, TensorGameError, _heads_to_slab, _slab_to_heads

SAVE_DIR_SYNTH_DEMOS = Path("data_unversioned/synthetic_demos")
SAVE_DIR_VAL = Path("data_unversioned/synthetic_demos_val")
SAVE_DIR_PLAYED_GAMES = Path("data_unversioned/played_games")
SAVE_DIR_BEST_GAMES = Path("data_unversioned/best_games")

PLAYED_GAMES_BUFFER_SIZE = 10000
BEST_GAMES_BUFFER_SIZE = 100

_STORE_NAME = "tg_demo_store.pt"


class SyntheticDemoDataset(Dataset):
    """datasets.py:20-158.  n_demos random rank-max_actions tensors with their action lists; item idx is
    (demo idx // max_actions, action idx % max_actions), demos being consumed last action first."""

    def __init__(self, max_actions: int, n_demos: int, dim_t: int, dim_3d: int, device: str, values=(-1, 0, 1),
                 probs=(0.15, 0.7, 0.15), shift=1, overwrite=True, save_dir=SAVE_DIR_SYNTH_DEMOS, **kwargs):
        super().__init__()
        self.max_actions = max_actions
        self.n_demos = n_demos
        self.dim_t = dim_t
        self.dim_3d = dim_3d
        self.values = torch.tensor(values)
        self.probs = torch.tensor(probs)
        self.shift = shift
        self.device = device
        self.save_dir = Path(save_dir)
        self.save_dir.mkdir(parents=True, exist_ok=True)
        self._cuda = _device()
        lay = _env.layout(dim_3d)
        store = self.save_dir / _STORE_NAME
        tape = torch.empty((max_actions, 0, lay.token_pitch), dtype=torch.uint8, device=self._cuda)
        slab = torch.empty((0, lay.game_pitch), dtype=torch.int8, device=self._cuda)
        if overwrite:
            for pattern in ("target_tensor_*.pt", "action_seq_*.pt", _STORE_NAME):
                for f in self.save_dir.glob(pattern):
                    f.unlink()
        else:
            tape, slab = self._load_existing(store, tape, slab)
        n_stored = slab.shape[0]
        if n_stored < n_demos:
            new_tape, new_slab = self._generate(n_demos - n_stored)
            tape = torch.cat((tape, new_tape), dim=1).contiguous()
            if new_slab.dtype != slab.dtype:  # one int16 target makes the whole store int16
                slab, new_slab = slab.to(torch.int16), new_slab.to(torch.int16)
            slab = torch.cat((slab, new_slab), dim=0).contiguous()
            torch.save({"tape": tape.cpu(), "slab": slab.cpu(), "max_actions": max_actions, "dim_3d": dim_3d,
                        "shift": shift}, store)
        # like the reference: more stored demos than asked for are simply not indexed (datasets.py:71-72)
        self._tape, self._slab = tape, slab
        # what __getitem__ reads: demo-major action records + targets (int8 slab, or int16 where a target left its zone)
        self._store = _env.DemoStore.from_tape(tape, slab, dim_3d, shift)

    # -- store ------------------------------------------------------------------------------------------
    def _load_existing(self, store: Path, tape, slab):
        if store.exists():
            blob = torch.load(store)
            if blob["max_actions"] == self.max_actions and blob["dim_3d"] == self.dim_3d:
                return blob["tape"].to(self._cuda), blob["slab"].to(self._cuda)
        # a directory written by the reference itself: one action_seq/target_tensor pair per demo
        n_ref = len(list(self.save_dir.glob("target_tensor_*.pt")))
        if n_ref:
            S = self.dim_3d
            toks = torch.stack([torch.stack(torch.load(self.save_dir / f"action_seq_{i}.pt")) for i in range(n_ref)])
            tgts = torch.stack([torch.load(self.save_dir / f"target_tensor_{i}.pt") for i in range(n_ref)])
            tape = _env.pack_actions(toks.reshape(-1, 3 * S).to(self._cuda), S).reshape(n_ref, self.max_actions, -1)
            tgts = tgts.to(self._cuda).float().contiguous()
            wide = bool(tgts.abs().max() > 63) if n_ref else False
            return tape.transpose(0, 1).contiguous(), (_env.pack_states16(tgts, S) if wide else _env.pack_states(tgts, S))
        return tape, slab

    def _generate(self, n: int):
        """n demos from torch's global CPU generator, exactly the stream the reference loop consumes."""
        tape, slab, flags, _ = _env.demos_from_seed(n, self.max_actions, self.dim_3d, self.values.tolist(),
                                                    self.probs.tolist(), self.shift, seed=None, device=self._cuda)
        if bool((flags & _env.FLAG_RANGE).any()):
            # a target left the int8 slab's zone (the reference accumulates in float32 without limit, utils.py:218-232):
            # the same action lists summed into the int16 format
            slab, f16 = _env.accumulate_demos16(tape, self.dim_3d, self.shift)
            if bool((f16 & _env.FLAG_RANGE).any()):
                raise TensorGameError("a synthetic target does not fit int16")
        return tape, slab

    # -- Dataset ----------------------------------------------------------------------------------------
    def __len__(self):
        return self.n_demos * self.max_actions

    def get_batch(self, indices):
        """Collated batch for many indices at once (one tg_demo_sample launch): states (B,T,S,S,S) f32,
        scalars (B,1) f32, actions (B,3S) i64, rewards (B,1) f32 on self.device."""
        idx = torch.as_tensor(indices, dtype=torch.int64).to(self._cuda)
        n_items = self._slab.shape[0] * self.max_actions
        if idx.numel() and (int(idx.min()) < 0 or int(idx.max()) >= n_items):
            raise IndexError(f"sample index out of range [0, {n_items})")
        # the reference replays with action_to_tensor, whose shift is fixed at 1 (SURVEY Q1)
        out = self._store.samples(idx, self.dim_t, replay_shift=1)
        return tuple(t.to(self.device) for t in out)

    @torch.no_grad()
    def __getitem__(self, idx: int):
        """datasets.py:77-122 -> (state (dim_t,S,S,S) f32, scalar (1,) f32, action (3S,) i64, reward (1,) f32)."""
        if not 0 <= idx < self._slab.shape[0] * self.max_actions:
            raise IndexError(idx)
        st, sc, ac, rw = self.get_batch([int(idx)])
        return st[0], sc[0], ac[0], rw[0]

    def __getitems__(self, indices):
        """DataLoader batched fetch: one kernel launch per batch instead of one per sample."""
        st, sc, ac, rw = self.get_batch(list(indices))
        return [(st[i], sc[i], ac[i], rw[i]) for i in range(len(indices))]

    def _create_synthetic_demos(self, n_demos_needed: int):
        """datasets.py:124-142: yields (action_seq list of (3S,) int64, target (S,S,S) float32)."""
        if n_demos_needed <= 0:
            return
        tape, slab = self._generate(n_demos_needed)
        S = self.dim_3d
        tokens = _env.unpack_actions(tape.reshape(-1, tape.shape[-1]), S).reshape(self.max_actions, n_demos_needed, 3 * S).cpu()
        targets = (_env.expand_states16(slab, S) if slab.dtype == torch.int16 else _env.expand_states(slab, S)).cpu()
        for d in range(n_demos_needed):
            yield [tokens[r, d] for r in range(self.max_actions)], targets[d]

    @staticmethod
    def _take_actions(action_seq: List[torch.Tensor], target_tensor: torch.Tensor):
        """datasets.py:144-153: target - sum of action_to_tensor(a) (shift fixed at 1), no early stop (tg_replay)."""
        if len(action_seq) == 0:
            return target_tensor
        S = target_tensor.shape[-1]
        dev = _device()
        tokens = torch.stack([a.reshape(-1) for a in action_seq]).to(dev).to(torch.int64)
        # coefficient = token - 1 (action_to_tensor's fixed shift, SURVEY Q1), re-based to (token + 3, shift 4) so that
        # the kernels' token bound holds for every alphabet the reference's datasets use
        tape = _env.pack_actions(tokens, S, rebase=_COEF_SHIFT - 1).unsqueeze(1)
        slab = _heads_to_slab(target_tensor.reshape(1, S, S, S), S)  # int8, or int16 for targets beyond it
        out, flags, _ = _env.replay(slab, tape, S, _COEF_SHIFT)
        if slab.dtype == torch.int8 and bool((flags & _env.FLAG_RANGE).any()):
            # the reference computes in float32 and never wraps: replay the int16 slab of the same values
            out, flags, _ = _env.replay(slab.to(torch.int16), tape, S, _COEF_SHIFT)
        if bool((flags & _env.FLAG_RANGE).any()):
            raise TensorGameError("_take_actions left the int16 slab's guaranteed range [-16384, 16383]")
        return _slab_to_heads(out, S, (), torch.float32, target_tensor.device)

    def _factor_sample(self):
        """datasets.py:155-158"""
        return self.values[Categorical(self.probs).sample(torch.Size([self.dim_3d]))]


class PlayedGamesDataset(Dataset):
    """datasets.py:161-230: ring buffer of played games (state, improved policy, reward per step).  The reference keeps
    three .pt files per game on disk; here the ring lives in HBM: states as int16 slabs (buffer_size, L, T, GP), policies
    float32 (buffer_size, L, n_steps, n_logits), rewards int64 (buffer_size, L), with L = the longest game seen (grown on
    demand).  Same ring semantics: game_pointer wraps at buffer_size and a new game overwrites the slot it lands on;
    items are indexed game by game in slot order."""

    def __init__(self, buffer_size: int, device: str, save_dir=SAVE_DIR_PLAYED_GAMES, **kwargs):
        super().__init__()
        self.game_pointer = 0
        self.buffer_size = buffer_size
        self.game_lengths = {}
        self.device = device
        self.save_dir = Path(save_dir)
        self.save_dir.mkdir(parents=True, exist_ok=True)
        self._states = self._policy = self._reward = None
        self._dims = None  # (T, S)

    def __del__(self):
        self._states = self._policy = self._reward = None
        self.game_pointer = 0

    def __len__(self):
        return sum(self.game_lengths.values())

    def _ensure(self, L: int, T: int, S: int, pol_shape):
        dev = _device()
        if self._states is None:
            lay = _env.layout(S)
            self._dims = (T, S)
            self._states = torch.zeros((self.buffer_size, L, T, lay.game_pitch), dtype=torch.int16, device=dev)
            self._policy = torch.zeros((self.buffer_size, L, *pol_shape), dtype=torch.float32, device=dev)
            self._reward = torch.zeros((self.buffer_size, L), dtype=torch.int64, device=dev)
        elif L > self._states.shape[1]:
            grow = lambda x: torch.cat((x, x.new_zeros((x.shape[0], L - x.shape[1], *x.shape[2:]))), dim=1)  # noqa: E731
            self._states, self._policy, self._reward = grow(self._states), grow(self._policy), grow(self._reward)
        if self._dims != (T, S) or tuple(self._policy.shape[2:]) != tuple(pol_shape):
            raise TensorGameError("PlayedGamesDataset: every game must have the same state and policy shape")

    def add_game(self, state_seq: List[torch.Tensor], action_seq: List[torch.Tensor], reward_seq: List[torch.Tensor]):
        n = len(state_seq)
        states = torch.stack([s.reshape(s.shape[-4:]) for s in state_seq]).to(torch.float32)  # (n, T, S, S, S)
        T, S = states.shape[1], states.shape[-1]
        policy = torch.stack([torch.as_tensor(a) for a in action_seq]).to(torch.float32) if not isinstance(action_seq, torch.Tensor) else action_seq.to(torch.float32)
        reward = torch.stack([torch.as_tensor(r).reshape(()) for r in reward_seq]) if not isinstance(reward_seq, torch.Tensor) else reward_seq
        self._ensure(n, T, S, policy.shape[1:])
        dev = self._states.device
        slab16 = _env.pack_states16(states.reshape(n * T, S, S, S).to(dev).contiguous(), S)
        g = self.game_pointer
        self._states[g, :n] = slab16.reshape(n, T, -1)
        self._policy[g, :n] = policy.to(dev)
        self._reward[g, :n] = reward.to(dev).to(torch.int64)
        self.game_lengths[g] = n
        self.game_pointer = (self.game_pointer + 1) % self.buffer_size

    def _locate(self, idx: int):
        i = 0
        while idx >= self.game_lengths[i]:
            idx -= self.game_lengths[i]
            i += 1
        return i, idx

    def get_batch(self, indices):
        """Collated items for many indices: one gather from the ring and one slab16 -> float32 expansion."""
        T, S = self._dims
        where = [self._locate(int(i)) for i in indices]
        dev = self._states.device
        g = torch.tensor([w[0] for w in where], dtype=torch.int64, device=dev)
        j = torch.tensor([w[1] for w in where], dtype=torch.int64, device=dev)
        slab16 = self._states[g, j].reshape(len(where) * T, -1).contiguous()
        states = _env.expand_states16(slab16, S).reshape(len(where), T, S, S, S)
        scalars = j.to(torch.float32).unsqueeze(1)                # get_scalars(state, idx, batch_size=False): the step index
        actions = self._policy[g, j].argmax(dim=-1)
        rewards = self._reward[g, j].unsqueeze(1)
        return tuple(t.to(self.device) for t in (states, scalars, actions, rewards))

    @torch.no_grad()
    def __getitem__(self, idx: int):
        st, sc, ac, rw = self.get_batch([idx])
        return st[0], sc[0], ac[0], rw[0]

    def __getitems__(self, indices):
        st, sc, ac, rw = self.get_batch(list(indices))
        return [(st[i], sc[i], ac[i], rw[i]) for i in range(len(indices))]


class TensorGameDataset(Dataset):
    """datasets.py:233-359: mixture of synthetic demos, played games and best games."""

    def __init__(self, len_data: int, fract_synth: float, max_actions: int, dim_t: int, dim_3d: int, device: str,
                 start_tensor=None, action_seq=None, **kwargs):
        super().__init__()
        self.len_data = len_data
        self.buffer_synth = SyntheticDemoDataset(max_actions, len_data, dim_t, dim_3d, device, **kwargs)
        self.buffer_played = PlayedGamesDataset(PLAYED_GAMES_BUFFER_SIZE, device, save_dir=SAVE_DIR_PLAYED_GAMES)
        self.buffer_best = PlayedGamesDataset(BEST_GAMES_BUFFER_SIZE, device, save_dir=SAVE_DIR_BEST_GAMES)
        self.is_synth = torch.ones(len_data, dtype=torch.bool)
        self.index_synth = torch.from_numpy(np.random.choice(len(self.buffer_synth), len_data, replace=False))
        self.index_played = None
        self.index_best = None
        self.fract_synth = fract_synth
        self.fract_best = 0
        self.dim_t = dim_t
        self.dim_3d = dim_3d
        self.device = device
        n = int(np.sqrt(dim_3d))
        if start_tensor is None:
            self.start_tensor = build_matmul_tensor(dim_t, n, n, n)
        else:
            self.start_tensor = start_tensor
            self.action_seq = action_seq

    def __len__(self):
        return self.len_data

    def _route(self, idx: int):
        """Which buffer and which index inside it serve dataset index idx (datasets.py:286-303)."""
        n_synth_before = int(self.is_synth[:idx].sum())
        if self.is_synth[idx]:
            return self.buffer_synth, int(self.index_synth[n_synth_before])
        rest = idx - n_synth_before
        if self.fract_best > 0 and self.index_best is not None:
            if rest < len(self.index_best):
                return self.buffer_best, int(self.index_best[rest])
            return self.buffer_played, int(self.index_played[rest - len(self.index_best)])
        return self.buffer_played, int(self.index_played[rest])

    def __getitem__(self, idx: int):
        buf, j = self._route(idx)
        return buf[j]

    def __getitems__(self, indices):
        """Batched fetch: the synthetic share of a batch is ONE tg_demo_sample launch."""
        routed = [self._route(int(i)) for i in indices]
        synth_pos = [p for p, (buf, _) in enumerate(routed) if buf is self.buffer_synth]
        out = [None] * len(routed)
        if synth_pos:
            items = self.buffer_synth.__getitems__([routed[p][1] for p in synth_pos])
            for p, item in zip(synth_pos, items):
                out[p] = item
        for other in (self.buffer_played, self.buffer_best):
            pos = [p for p, (buf, _) in enumerate(routed) if buf is other]
            if pos:
                for p, item in zip(pos, other.__getitems__([routed[p][1] for p in pos])):
                    out[p] = item
        return out

    def set_fractions(self, fract_synth, fract_best):
        self.fract_synth = fract_synth
        self.fract_best = fract_best

    def resample_buffer_indexes(self):
        """datasets.py:310-343, including int(1 - fs - fb) * len_data == 0 for positive fractions (SURVEY Q10)."""
        if len(self.buffer_played) == 0:
            return
        self.is_synth = torch.rand(self.len_data) < self.fract_synth
        len_synth = self.is_synth.sum().item()
        self.index_synth = torch.from_numpy(np.random.choice(len(self.buffer_synth), len_synth, replace=False))
        if len(self.buffer_best) > 0 and self.fract_best > 0:
            len_played = int(1 - self.fract_synth - self.fract_best) * self.len_data
            len_best = self.len_data - len_synth - len_played
            self.index_played = torch.from_numpy(
                np.random.choice(len(self.buffer_played), len_played, replace=len_played > len(self.buffer_played)))
            self.index_best = torch.from_numpy(
                np.random.choice(len(self.buffer_best), len_best, replace=len_best > len(self.buffer_best)))
        else:
            len_played = self.len_data - len_synth
            self.index_played = torch.from_numpy(
                np.random.choice(len(self.buffer_played), len_played, replace=len_played > len(self.buffer_played)))

    def add_played_game(self, state_seq, action_seq, reward_seq):
        self.buffer_played.add_game(state_seq, action_seq, reward_seq)

    def add_best_game(self, state_seq, action_seq, reward_seq):
        self.buffer_best.add_game(state_seq, action_seq, reward_seq)


class StrassenDemoDataset(Dataset):
    """datasets.py:362-420: every (state, next action) pair over all 2^7 subsets of Strassen's seven products;
    448 items, states (1,4,4,4) float32, actions = factors + 2, reward = -#unused products, scalar 0.
    The 128 subset states are one tg_demo_accumulate launch (state = sum of the UNUSED products)."""

    def __init__(self, max_len=None):
        self.n_total = 7
        self.device = "cpu"
        uu, vv, ww = get_strassen_factors(self.device)
        factors = torch.cat((uu, vv, ww), dim=1)  # (7, 12)
        codes = torch.arange(2 ** self.n_total)
        used = ((codes.unsqueeze(1) >> (self.n_total - 1 - torch.arange(self.n_total))) & 1).bool()  # MSB = product 0
        # tape (7, 128, TP): step r of subset s carries product r if unused, the null action otherwise
        tok = torch.where(used.t().unsqueeze(-1), torch.zeros_like(factors).unsqueeze(1), factors.unsqueeze(1)) + _COEF_SHIFT
        dev = _device()
        tape = _env.pack_actions(tok.reshape(-1, 12).to(dev), 4).reshape(self.n_total, 2 ** self.n_total, -1)
        slab, _ = _env.accumulate_demos(tape, 4, _COEF_SHIFT)
        states = _env.expand_states(slab, 4).cpu()
        self.state_tensor, self.target_action, self.reward, self.scalar, self.bit_info = [], [], [], [], []
        for s in range(2 ** self.n_total):
            avail = [r for r in range(self.n_total) if not used[s, r]]
            for r in avail:
                self.state_tensor.append(states[s].unsqueeze(0))
                self.target_action.append(factors[r] + 2)
                self.reward.append(torch.tensor([-len(avail)], dtype=torch.float32))
                self.scalar.append(torch.tensor([0.0], dtype=torch.float32))
                self.bit_info.append(format(s, "b").zfill(self.n_total))
        self.n_demos = len(self.state_tensor)
        if max_len:
            self.state_tensor = self.state_tensor[:max_len]
            self.target_action = self.target_action[:max_len]
            self.reward = self.reward[:max_len]
            self.scalar = self.scalar[:max_len]
            self.n_demos = max_len

    def __len__(self):
        return self.n_demos

    @torch.no_grad()
    def __getitem__(self, idx: int):
        return (self.state_tensor[idx].to(self.device), self.scalar[idx].to(self.device),
                self.target_action[idx].to(self.device), self.reward[idx].to(self.device))


def _signs(rows):
    return torch.tensor([[{"+": 1, "-": -1, "0": 0}[c] for c in row] for row in rows])


def get_strassen_factors(device: str):
    """datasets.py:423-460: Strassen's seven products as (u, v, w) factor rows over vec(A), vec(B), vec(C)."""
    uu = _signs(["+00+", "00++", "+000", "000+", "++00", "-0+0", "0+0-"])
    vv = _signs(["+00+", "+000", "0+0-", "-0+0", "000+", "++00", "00++"])
    ww = _signs(["+00+", "00+-", "0+0+", "+0+0", "-+00", "000+", "+000"])
    return uu.to(device), vv.to(device), ww.to(device)


def get_strassen_tensor(device: str):
    """datasets.py:463-465"""
    return uvw_to_demo(*get_strassen_factors(device), device)
