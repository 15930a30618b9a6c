"""Exact 2x2x2 distances (TEST INFRASTRUCTURE ONLY -- see oracle/__init__.py): the spec of include/cube_b200.h
cube_distance_* that the tests compare the CUDA path against.

rank = L * 729 + T over py222 getOP (p_i, o_i) of slots 0..6: L = the Lehmer code of p, T = o_0..o_5 in base 3
(o_6 is implied).  A row is reachable exactly when the row rebuilt from its rank is the row.
"""
import numpy as np

from . import tables as T
from .cube_np import apply_moves, decode_2, get_op, solved_states

DISTANCE_ENTRIES_2 = 5040 * 729
UNREACHABLE = 255
_FACT = np.array([720, 120, 24, 6, 2, 1, 1], dtype=np.int64)


def _rank_of_op(p, o):
    r = np.zeros(len(p), dtype=np.int64)
    for i in range(7):
        r += (p[:, i + 1:] < p[:, i:i + 1]).sum(axis=1) * _FACT[i]
    t = np.zeros(len(p), dtype=np.int64)
    for i in range(6):
        t = t * 3 + o[:, i]
    return r * 729 + t


def unrank_2(ranks):
    """Sticker rows [N, 24] uint8 of ranks [N] (every rank is a reachable state)."""
    ranks = np.asarray(ranks, dtype=np.int64)
    n = len(ranks)
    lehmer, t = ranks // 729, ranks % 729
    o = np.zeros((n, 7), dtype=np.int64)
    for i in range(5, -1, -1):
        o[:, i], t = t % 3, t // 3
    o[:, 6] = (-o[:, :6].sum(axis=1)) % 3
    p = np.zeros((n, 7), dtype=np.int64)
    free = np.tile(np.arange(7), (n, 1))
    for i in range(7):
        d, lehmer = lehmer // _FACT[i], lehmer % _FACT[i]
        p[:, i] = free[np.arange(n), d]
        free = np.where(np.arange(7 - i)[None, :-1] >= d[:, None], free[:, 1:], free[:, :-1])
    cols = np.zeros((n, 7, 21), dtype=np.uint8)                     # the one-hot rows decode_2 inverts
    cols[np.arange(n)[:, None], p, 3 * np.arange(7)[None, :] + o] = 1
    return decode_2(cols)


def rank_2(states):
    """Rank of every 2x2x2 sticker row [N, 24], -1 where the row is not reachable."""
    states = np.asarray(states, dtype=np.uint8)
    h = states[:, T.PIECE_DEFS_2].astype(np.int64) @ T.HASH_W_2
    valid = (h < len(T.PIECE_INDS_2)).all(axis=1)                    # else a hash outside py222's table
    s = np.where(valid[:, None], states, T.SOLVED[2][None, :]).astype(np.uint8)
    op = get_op(2, s)
    r = _rank_of_op(op[:, :, 0], op[:, :, 1])
    valid &= (unrank_2(r) == states).all(axis=1)
    return np.where(valid, r, -1)


def distance_table_2():
    """uint8 [3 674 160]: the quarter-turn distance of every rank, by breadth-first search from solved."""
    dist = np.full(DISTANCE_ENTRIES_2, UNREACHABLE, dtype=np.uint8)
    front = solved_states(2, 1)
    dist[rank_2(front)] = 0
    d = 0
    while len(front):
        kids = np.concatenate([apply_moves(2, front, np.full(len(front), a)) for a in range(6)])
        op = get_op(2, kids)
        r, idx = np.unique(_rank_of_op(op[:, :, 0], op[:, :, 1]), return_index=True)
        new = dist[r] == UNREACHABLE
        d += 1
        dist[r[new]] = d
        front = kids[idx[new]]
    return dist


def distance_2(table, states):
    """table[rank] of every row, 255 where unreachable."""
    r = rank_2(states)
    return np.where(r >= 0, table[np.maximum(r, 0)], UNREACHABLE).astype(np.uint8)


def solve_optimal_2(table, states, max_len=14):
    """(actions [N, 14] uint8 padded with the no-op index 12, length [N] uint8): at every step the lowest action
    index whose child is one level closer; length 255 and only no-ops for an unreachable row."""
    states = np.array(states, dtype=np.uint8)
    n = len(states)
    actions = np.full((n, max_len), 12, dtype=np.uint8)
    d = distance_2(table, states).astype(np.int64)
    length = d.astype(np.uint8)
    for k in range(max_len):
        live = np.flatnonzero((d > 0) & (d != UNREACHABLE))
        if not len(live):
            break
        kids = np.stack([apply_moves(2, states[live], np.full(len(live), a)) for a in range(6)], axis=1)
        kd = distance_2(table, kids.reshape(-1, 24)).reshape(len(live), 6).astype(np.int64)
        a = (kd == d[live, None] - 1).argmax(axis=1)
        actions[live, k] = a
        states[live] = kids[np.arange(len(live)), a]
        d[live] -= 1
    return actions, length
