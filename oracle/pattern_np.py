"""3x3x3 pattern databases (TEST INFRASTRUCTURE ONLY -- see oracle/__init__.py): the spec of include/cube_b200.h
cube_pattern_* / cube_distance_bound / cube_solve_bounded that the tests compare the CUDA path against, and an
exact distance that needs no pattern database at all.

Cubies are the exact encoding's (piece, ori) per slot (cube_np.onehot_columns_exact): corners 3 * piece + ori,
edges 2 * piece + ori.  Sections of the table buffer, one byte per rank:
  corners  Lehmer(p_0..p_7) * 2187 + sum_{q<7} o_q * 3^(6-q)
  edges A  pieces k = 0..5: slot of piece k counted among the slots not yet taken, mixed radix 12 * 11 * .. * 7,
           then * 64 + the six flips in base 2 (piece 0 the most significant)
  edges B  the same for pieces 6..11 with slots relabelled s -> (s - 6) mod 12
"""
import numpy as np

from . import tables as T
from .cube_np import apply_moves, decode_exact, solved_states

CORNERS, EDGES = 88179840, 42577920
OFFSETS = (0, CORNERS, CORNERS + EDGES)
ENTRIES = (CORNERS, EDGES, EDGES)
TABLES_BYTES = CORNERS + 2 * EDGES
UNREACHABLE = 255
_FACT8 = np.array([5040, 720, 120, 24, 6, 2, 1, 1], dtype=np.int64)


def _columns(states):
    """[N, 20] exact one-hot columns of sticker rows whose colours are < 6 (any hash: an unassigned one gives a
    column whose rebuilt stickers differ from the row)."""
    from .cube_np import CORNER_DEFS_EXACT, CORNER_INDS_EXACT
    s = states.astype(np.int64)
    hc = s[:, CORNER_DEFS_EXACT] @ T.CORNER_HASH_W
    op = CORNER_INDS_EXACT[np.minimum(hc, len(CORNER_INDS_EXACT) - 1)]
    he = s[:, T.EDGE_DEFS_3] @ T.EDGE_HASH_W
    eo = T.EDGE_INDS_3[np.minimum(he, len(T.EDGE_INDS_3) - 1)]
    cols = np.empty((len(s), 20), dtype=np.int64)
    cols[:, :8] = np.maximum(op[:, :, 0], 0) * 3 + np.maximum(op[:, :, 1], 0)
    cols[:, 8:] = eo[:, :, 0] * 2 + eo[:, :, 1]
    return cols


def _parity(p):
    n = p.shape[1]
    inv = sum((p[:, i + 1:] < p[:, i:i + 1]).sum(axis=1) for i in range(n))
    return inv & 1


def cubies(states):
    """(corner piece [N, 8], corner ori [N, 8], edge piece [N, 12], edge ori [N, 12], reachable [N]).  A row is
    reachable when the row rebuilt from its cubies is the row (centres, colours), the pieces are permutations, the
    twists sum to 0 mod 3, the flips to 0 mod 2 and the corner and edge permutations have the same parity."""
    states = np.asarray(states, dtype=np.uint8)
    ok = (states < 6).all(axis=1)
    s = np.where(ok[:, None], states, solved_states(3, 1)).astype(np.uint8)
    cols = _columns(s)
    onehot = np.zeros((len(s), 20, 24), dtype=np.uint8)
    onehot[np.arange(len(s))[:, None], np.arange(20)[None, :], cols] = 1
    ok &= (decode_exact(onehot) == s).all(axis=1)
    cp, co, ep, eo = cols[:, :8] // 3, cols[:, :8] % 3, cols[:, 8:] // 2, cols[:, 8:] % 2
    ok &= (np.sort(cp, axis=1) == np.arange(8)).all(axis=1) & (np.sort(ep, axis=1) == np.arange(12)).all(axis=1)
    ok &= (co.sum(axis=1) % 3 == 0) & (eo.sum(axis=1) % 2 == 0) & (_parity(cp) == _parity(ep))
    return cp, co, ep, eo, ok


def rank_corners(p, o):
    lehmer = sum((p[:, i + 1:] < p[:, i:i + 1]).sum(axis=1) * _FACT8[i] for i in range(8))
    t = np.zeros(len(p), dtype=np.int64)
    for q in range(7):
        t = t * 3 + o[:, q]
    return lehmer * 2187 + t


def unrank_corners(ranks):
    ranks = np.asarray(ranks, dtype=np.int64)
    n = len(ranks)
    lehmer, t = ranks // 2187, ranks % 2187
    o = np.zeros((n, 8), dtype=np.int64)
    for q in range(6, -1, -1):
        o[:, q], t = t % 3, t // 3
    o[:, 7] = (-o[:, :7].sum(axis=1)) % 3
    p = np.zeros((n, 8), dtype=np.int64)
    free = np.tile(np.arange(8), (n, 1))
    for i in range(8):
        d, lehmer = lehmer // _FACT8[i], lehmer % _FACT8[i]
        p[:, i] = free[np.arange(n), d]
        free = np.where(np.arange(8 - i)[None, :-1] >= d[:, None], free[:, 1:], free[:, :-1])
    return p, o


def rank_edges(slot, flip):
    """slot [N, 6]: the (relabelled) slot of tracked piece k = 0..5; flip [N, 6]: its flip."""
    r = np.zeros(len(slot), dtype=np.int64)
    for k in range(6):
        r = r * (12 - k) + slot[:, k] - (slot[:, :k] < slot[:, k:k + 1]).sum(axis=1)
    f = np.zeros(len(slot), dtype=np.int64)
    for k in range(6):
        f = f * 2 + flip[:, k]
    return r * 64 + f


def unrank_edges(ranks):
    ranks = np.asarray(ranks, dtype=np.int64)
    n = len(ranks)
    f, r = ranks % 64, ranks // 64
    digit = np.zeros((n, 6), dtype=np.int64)
    for k in range(5, -1, -1):
        digit[:, k], r = r % (12 - k), r // (12 - k)
    flip = np.stack([(f >> (5 - k)) & 1 for k in range(6)], axis=1)
    slot = np.zeros((n, 6), dtype=np.int64)
    free = np.tile(np.arange(12), (n, 1))
    for k in range(6):
        slot[:, k] = free[np.arange(n), digit[:, k]]
        free = np.where(np.arange(12 - k)[None, :-1] >= digit[:, k:k + 1], free[:, 1:], free[:, :-1])
    return slot, flip


def _edge_section(ep, eo, base):
    where = np.argsort(ep, axis=1)                              # slot of every piece
    slot = where[:, base:base + 6]
    flip = np.take_along_axis(eo, slot, axis=1)
    return rank_edges((slot - base) % 12, flip)


def ranks(states):
    """[N, 3] ranks (corners, edges A, edges B) of sticker rows; -1 in every column of an unreachable row."""
    cp, co, ep, eo, ok = cubies(states)
    r = np.stack([rank_corners(cp, co), _edge_section(ep, eo, 0), _edge_section(ep, eo, 6)], axis=1)
    return np.where(ok[:, None], r, -1)


def bound(tables, states, parts=False):
    """cube_distance_bound: max of the three section values, plus 1 when its parity differs from the corner
    permutation's; 255 (and parts of 255) for an unreachable row."""
    cp, _, _, _, ok = cubies(states)
    r = ranks(states)
    h = np.stack([tables[OFFSETS[k] + np.maximum(r[:, k], 0)] for k in range(3)], axis=1).astype(np.int64)
    b = h.max(axis=1)
    b += (b ^ _parity(cp)) & 1
    b = np.where(ok, b, UNREACHABLE).astype(np.uint8)
    h = np.where(ok[:, None], h, UNREACHABLE).astype(np.uint8)
    return (b, h) if parts else b


# ---- an exact distance without pattern databases: meet in the middle ----------------------------------------
def _keys(states):
    """One exact key per reachable state: corner rank * EDGES + edges-A rank (< 2^52) as the real part, the edges-B
    rank as the imaginary part of a complex128.  Both are exact in float64, and NumPy sorts and searches complex
    numbers lexicographically, so sorted keys can be searched in one call."""
    r = ranks(states)
    assert (r >= 0).all(), "keys of unreachable rows"
    return (r[:, 0] * EDGES + r[:, 1]).astype(np.float64) + 1j * r[:, 2].astype(np.float64)


class Ball(object):
    """Every state within `radius` quarter turns of solved, as sorted keys with their distances; level_sizes[d] =
    the number of states at distance d (1, 12, 114, 1 068, 10 011, 93 840, 878 880)."""

    def __init__(self, radius=6):
        self.radius = radius
        front = solved_states(3, 1)
        keys, dist, self.level_sizes = [_keys(front)], [np.zeros(1, dtype=np.int64)], [1]
        seen = np.sort(keys[0])
        for d in range(1, radius + 1):
            kids = np.concatenate([apply_moves(3, front, np.full(len(front), a)) for a in range(12)])
            k = _keys(kids)
            k, idx = np.unique(k, return_index=True)
            pos = np.minimum(np.searchsorted(seen, k), len(seen) - 1)
            new = seen[pos] != k
            front, k = kids[idx[new]], k[new]
            keys.append(k)
            dist.append(np.full(len(k), d, dtype=np.int64))
            self.level_sizes.append(len(k))
            seen = np.sort(np.concatenate([seen, k]))
        k, d = np.concatenate(keys), np.concatenate(dist)
        order = np.argsort(k)
        self.keys, self.dist = k[order], d[order]

    def lookup(self, keys):
        """Distance from solved of every key, -1 where the key is outside the ball."""
        pos = np.minimum(np.searchsorted(self.keys, keys), len(self.keys) - 1)
        return np.where(self.keys[pos] == keys, self.dist[pos], -1)


def exact_distance(ball, states, max_radius=6, chunk=256):
    """The quarter-turn distance of every reachable row: the states k turns from the row, k = 0, 1, ..., met with
    the ball around solved.  best_k = min over those of k + distance from solved is an upper bound, and the exact
    distance d once best_k <= k + ball.radius (an optimal path then has a state within the ball at most k turns
    from the row).  Rows needing more than max_radius turns from their side raise."""
    states = np.asarray(states, dtype=np.uint8)
    out = np.empty(len(states), dtype=np.int64)
    for lo in range(0, len(states), chunk):
        rows = states[lo:lo + chunk]
        n = len(rows)
        best = np.full(n, 1 << 30, dtype=np.int64)
        done = np.zeros(n, dtype=bool)
        front, qid, last = rows, np.arange(n), np.full(n, -1)
        for k in range(max_radius + 1):
            d0 = ball.lookup(_keys(front))
            hit = d0 >= 0
            np.minimum.at(best, qid[hit], k + d0[hit])
            done |= best <= k + ball.radius
            if done.all():
                break
            live = ~done[qid]
            front, qid, last = front[live], qid[live], last[live]
            kids, kq, kl = [], [], []
            for a in range(12):                                 # never undo the move just made
                sel = last != (a ^ 1)
                kids.append(apply_moves(3, front[sel], np.full(int(sel.sum()), a)))
                kq.append(qid[sel])
                kl.append(np.full(int(sel.sum()), a))
            front, qid, last = np.concatenate(kids), np.concatenate(kq), np.concatenate(kl)
        assert done.all(), "a row is farther than the ball and max_radius reach"
        out[lo:lo + n] = best
    return out
