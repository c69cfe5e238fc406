"""numpy reference for the mod-2 training samples (include/tensorgame.h "mod-2 training samples"): the batch
tg_demo_sample_gf2 writes from a demo-major store with bit-slab targets.  States are 0/1; a token t stands for the
residue (t - replay_shift) & 1."""
import numpy as np

from tests import gf2_ref


def demo_getitem(tok, target, dim_t: int, a: int, replay_shift: int) -> np.ndarray:
    """tok (R, 3S), target (S,S,S) integers -> states (dim_t,S,S,S) 0/1: slot 0 = target xor the terms of records
    a+1 .. R-1, slot t = the term of record min(a + dim_t, R) - t where that is after a, else zero."""
    tok = np.asarray(tok, dtype=np.int64)
    R, S = tok.shape[0], tok.shape[1] // 3
    state = np.zeros((dim_t, S, S, S), dtype=np.int64)
    state[0] = (np.asarray(target, dtype=np.int64) & 1) ^ np.bitwise_xor.reduce(gf2_ref.rank1(tok[a + 1:], replay_shift), axis=0,
                                                                                  initial=0)
    hi = min(a + dim_t, R)
    for t in range(1, dim_t):
        if hi - t > a:
            state[t] = gf2_ref.rank1(tok[hi - t], replay_shift)
    return state


def samples(tok, targets, idx, dim_t: int, replay_shift: int):
    """tok (N, R, 3S), targets (N,S,S,S), idx (nb,) -> (states uint8 0/1 (nb,dim_t,S,S,S), scalars, actions, rewards,
    valid): demo_getitem of every sample, from per-demo suffix xors.  An index outside [0, N R) has zero states; its
    scalars, actions and rewards are not defined (valid False)."""
    tok = np.asarray(tok, dtype=np.int64)
    N, R, S = tok.shape[0], tok.shape[1], tok.shape[2] // 3
    idx = np.asarray(idx, dtype=np.int64)
    nb = idx.shape[0]
    terms = gf2_ref.rank1(tok, replay_shift).astype(np.uint8)                     # (N, R, S, S, S)
    after = np.zeros_like(terms)                                                  # after[d, a] = xor of terms a+1 .. R-1
    after[:, : R - 1] = np.bitwise_xor.accumulate(terms[:, :0:-1], axis=1)[:, ::-1]
    valid = (idx >= 0) & (idx < N * R)
    d, a = np.divmod(np.where(valid, idx, 0), R)
    states = np.zeros((nb, dim_t, S, S, S), dtype=np.uint8)
    states[:, 0] = (np.asarray(targets, dtype=np.int64)[d] & 1).astype(np.uint8) ^ after[d, a]
    hi = np.minimum(a + dim_t, R)
    for t in range(1, dim_t):
        j = hi - t
        states[:, t] = np.where((j > a)[:, None, None, None], terms[d, np.maximum(j, 0)], 0)
    states[~valid] = 0
    scalars = (R - a).astype(np.float32)[:, None]
    rewards = (-(a + 1)).astype(np.float32)[:, None]
    return states, scalars, tok[d, a], rewards, valid
