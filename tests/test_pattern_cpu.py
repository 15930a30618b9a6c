"""The 3x3x3 pattern databases without a GPU: the oracle's ranks and reachability, the per-state code of the pattern
kernels (csrc/cube_pattern.cuh compiled with g++ by tests/host_emul/pattern_emul.cpp) against the oracle, the
emulated build of the three tables against their known level counts and digests, the bound and the bounded IDA*
solve against an exact distance that uses no pattern database (meet in the middle), and the C ABI's argument
checks."""
import ctypes
import hashlib
import os
import subprocess
import threading

import numpy as np
import pytest

from oracle import cube_np as O
from oracle import pattern_np as P
from oracle import tables as T

HERE = os.path.dirname(os.path.abspath(__file__))

# states per quarter-turn distance of each section's pattern, and each section's digest (rank order)
LEVELS = [
    [1, 12, 114, 924, 6539, 39528, 199926, 806136, 2761740, 8656152, 22334112, 32420448, 18780864, 2166720, 6624],
    [1, 12, 109, 941, 7767, 60751, 439746, 2768420, 12518862, 22465564, 4312983, 2764],
    [1, 10, 93, 832, 6904, 54904, 406895, 2646406, 12435645, 22838844, 4185743, 1643],
]
SHA256 = ["b08ee2f4382a4987021e02ece8f1bb7908ae792a9059881ed4275222e321d0a7",
          "2323902f21856c0484551be789ac2e339ffcb57370538ad4c68709e526e1b3f9",
          "df9cfffdd423f96167ba8a07949ca40cb5df4280c8cdaddc1ccd79a6e4fbe289"]


def scrambles(n, seed, max_depth):
    """n sticker rows scrambled from solved, depths 0..max_depth (uniform)."""
    rng = np.random.RandomState(seed)
    moves = rng.randint(12, size=(n, max_depth)).astype(np.uint8)
    depth = rng.randint(0, max_depth + 1, size=n)
    out = np.empty((n, 54), dtype=np.uint8)
    for d in np.unique(depth):
        out[depth == d] = O.scramble(3, moves[depth == d, :d])
    return out


def garbage(seed, per_kind=100):
    """Rows that are no reachable state, per_kind of each: random bytes, a colour >= 6, two stickers of different
    colours swapped, a twisted corner, a flipped edge, two edges swapped (a parity error), a moved centre."""
    rng = np.random.RandomState(seed)
    good = scrambles(6 * per_kind, seed + 1, 25)
    k = per_kind
    idx = np.arange(k)[:, None]
    rnd = rng.randint(0, 256, size=(k, 54)).astype(np.uint8)
    colour = good[:k].copy()
    colour[np.arange(k), rng.randint(54, size=k)] = rng.randint(6, 256, size=k)
    swapped = good[k:2 * k].copy()
    for row in swapped:
        i, j = rng.choice(54, size=2, replace=False)
        while row[i] == row[j]:
            i, j = rng.choice(54, size=2, replace=False)
        row[i], row[j] = row[j], row[i]
    twisted = good[2 * k:3 * k].copy()
    slots = O.CORNER_DEFS_EXACT[rng.randint(8, size=k)]
    twisted[idx, slots] = twisted[idx, np.roll(slots, 1, axis=1)]
    flipped = good[3 * k:4 * k].copy()
    slots = T.EDGE_DEFS_3[rng.randint(12, size=k)]
    flipped[idx, slots] = flipped[idx, slots[:, ::-1]]
    parity = good[4 * k:5 * k].copy()
    pairs = np.array([rng.choice(12, size=2, replace=False) for _ in range(k)])
    a, b = T.EDGE_DEFS_3[pairs[:, 0]], T.EDGE_DEFS_3[pairs[:, 1]]
    parity[idx, a], parity[idx, b] = good[4 * k:5 * k][idx, b], good[4 * k:5 * k][idx, a]
    centre = good[5 * k:6 * k].copy()
    faces = np.array([rng.choice(6, size=2, replace=False) for _ in range(k)])
    centre[idx, 9 * faces + 4] = centre[idx, 9 * faces[:, ::-1] + 4]
    return [rnd, colour, swapped, twisted, flipped, parity, centre]


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    lib_path = str(tmp_path_factory.mktemp("pattern_emul") / "libpattern_emul.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-pthread", "-w", "-o", lib_path,
                           os.path.join(HERE, "host_emul", "pattern_emul.cpp")])
    lib = ctypes.CDLL(lib_path)
    vp, ll, ci = ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int
    for name in ("emul_pat3_bytes", "emul_pat3_offset", "emul_pat3_entries", "emul_pat3_roundtrip_failures",
                 "emul_pat3_check"):
        getattr(lib, name).restype = ll
    lib.emul_pat3_offset.argtypes = [ci]
    lib.emul_pat3_entries.argtypes = [ci]
    lib.emul_pat3_rank.argtypes = [vp, ll, vp, vp]
    lib.emul_pat3_child_ranks.argtypes = [vp, ll, vp]
    lib.emul_pat3_roundtrip_failures.argtypes = [ci, ll]
    lib.emul_pat3_build.argtypes = [vp, ci]
    lib.emul_pat3_check.argtypes = [vp, ci, ci]
    lib.emul_pat3_bound.argtypes = [vp, vp, ll, vp, vp]
    lib.emul_pat3_solve.argtypes = [vp, vp, ll, ci, ll, vp, vp, vp, vp]
    return lib


@pytest.fixture(scope="module")
def tables(emul):
    """The emulated build: the three sections in parallel threads (ctypes releases the GIL)."""
    t = np.empty(P.TABLES_BYTES, dtype=np.uint8)
    workers = [threading.Thread(target=emul.emul_pat3_build, args=(_p(t), s)) for s in range(3)]
    for w in workers:
        w.start()
    for w in workers:
        w.join()
    return t


@pytest.fixture(scope="module")
def ball():
    return P.Ball(6)


def emul_solve(emul, tables, rows, max_length, max_nodes, threads=8):
    rows = np.ascontiguousarray(rows)
    n = len(rows)
    actions = np.empty((n, max_length), dtype=np.uint8)
    length, lower = np.empty(n, dtype=np.uint8), np.empty(n, dtype=np.uint8)
    nodes = np.empty(n, dtype=np.int64)
    cuts = np.linspace(0, n, threads + 1).astype(int)

    def part(lo, hi):
        emul.emul_pat3_solve(_p(tables), _p(rows[lo:]), hi - lo, max_length, max_nodes,
                             _p(actions[lo:]), _p(length[lo:]), _p(lower[lo:]), _p(nodes[lo:]))
    workers = [threading.Thread(target=part, args=(cuts[i], cuts[i + 1])) for i in range(threads)]
    for w in workers:
        w.start()
    for w in workers:
        w.join()
    return actions, length, lower, nodes


def emul_bound(emul, tables, rows):
    rows = np.ascontiguousarray(rows)
    bound, parts = np.empty(len(rows), dtype=np.uint8), np.empty((len(rows), 3), dtype=np.uint8)
    emul.emul_pat3_bound(_p(tables), _p(rows), len(rows), _p(bound), _p(parts))
    return bound, parts


def walk(rows, actions):
    end = rows.copy()
    for k in range(actions.shape[1]):
        live = actions[:, k] < 12
        end[live] = O.apply_moves(3, end[live], actions[live, k])
    return end


# ---- the oracle ---------------------------------------------------------------------------------------------
def test_oracle_rank_round_trips_and_solved_rank():
    rng = np.random.RandomState(0)
    r = rng.randint(0, P.CORNERS, size=20000)
    assert (P.rank_corners(*P.unrank_corners(r)) == r).all()
    r = rng.randint(0, P.EDGES, size=20000)
    assert (P.rank_edges(*P.unrank_edges(r)) == r).all()
    assert (P.ranks(O.solved_states(3, 1)) == 0).all()
    assert P.OFFSETS == (0, 88179840, 130757760) and P.TABLES_BYTES == 173335680
    assert all(o % 16 == 0 for o in P.OFFSETS)


def test_ball_sizes_are_the_published_counts(ball):
    assert ball.level_sizes == [1, 12, 114, 1068, 10011, 93840, 878880]          # OEIS A080629


def test_reachable_and_unreachable_rows(emul):
    good = np.concatenate([scrambles(3000, 1, 40), O.solved_states(3, 1)])
    assert P.cubies(good)[4].all() and (P.ranks(good) >= 0).all()
    for rows in garbage(2):
        assert not P.cubies(rows)[4].any() and (P.ranks(rows) == -1).all()
        got_r, ok = np.empty((len(rows), 3), dtype=np.int64), np.empty(len(rows), dtype=np.uint8)
        emul.emul_pat3_rank(_p(np.ascontiguousarray(rows)), len(rows), _p(got_r), _p(ok))
        assert not ok.any()


# ---- the per-state code on the CPU ---------------------------------------------------------------------------
def test_emulated_ranks_and_turns(emul):
    assert emul.emul_pat3_bytes() == P.TABLES_BYTES
    assert [emul.emul_pat3_offset(s) for s in range(3)] == list(P.OFFSETS)
    assert [emul.emul_pat3_entries(s) for s in range(3)] == list(P.ENTRIES)
    assert [emul.emul_pat3_roundtrip_failures(s, 997) for s in range(3)] == [0, 0, 0]
    rows = np.ascontiguousarray(scrambles(20000, 3, 40))
    got, ok = np.empty((len(rows), 3), dtype=np.int64), np.empty(len(rows), dtype=np.uint8)
    emul.emul_pat3_rank(_p(rows), len(rows), _p(got), _p(ok))
    assert ok.all() and (got == P.ranks(rows)).all()
    rows = rows[:3000].copy()
    kids = np.empty((len(rows), 12, 3), dtype=np.int64)
    emul.emul_pat3_child_ranks(_p(rows), len(rows), _p(kids))
    children, _ = O.expand(3, rows)
    assert (kids == P.ranks(children.reshape(-1, 54)).reshape(len(rows), 12, 3)).all()


def test_emulated_build_is_the_bfs_distance_table(emul, tables):
    for s in range(3):
        sec = tables[P.OFFSETS[s]:P.OFFSETS[s] + P.ENTRIES[s]]
        assert np.bincount(sec, minlength=256).tolist() == LEVELS[s] + [0] * (256 - len(LEVELS[s]))
        assert hashlib.sha256(sec.tobytes()).hexdigest() == SHA256[s]
    assert [emul.emul_pat3_check(_p(tables), s, 8) for s in range(3)] == [0, 0, 0]


def test_bound_and_bounded_solve_against_the_exact_distance(emul, tables, ball):
    rows = scrambles(2000, 4, 10)
    exact = P.exact_distance(ball, rows)
    bound, parts = emul_bound(emul, tables, rows)
    want_b, want_p = P.bound(tables, rows, parts=True)
    assert (bound == want_b).all() and (parts == want_p).all()
    assert (bound <= exact).all() and ((exact - bound) % 2 == 0).all() and (bound[exact == 0] == 0).all()
    actions, length, lower, nodes = emul_solve(emul, tables, rows, 14, 1 << 40)
    assert (length == exact).all() and (lower == exact).all()
    assert ((actions < 12).sum(axis=1) == length).all()
    for k in range(14):                                                  # the NOOP padding comes after the solution
        assert ((actions[:, k] < 12) == (k < length)).all()
    assert O.is_solved(3, walk(rows, actions)).all()
    assert (nodes[exact == 0] == 0).all() and (nodes[exact > 0] > 0).all()
    # a budget below what the search needs: unproven, with a lower bound that still holds
    hard = np.flatnonzero(nodes > 1)
    _, l2, lo2, n2 = emul_solve(emul, tables, rows[hard], 14, 1)
    assert (l2 == 255).all() and (lo2 <= exact[hard]).all() and (n2 == 1).all()
    half = nodes[hard] // 2
    for i in np.flatnonzero(hard)[:200]:
        _, l3, lo3, n3 = emul_solve(emul, tables, rows[hard[i]:hard[i] + 1], 14, int(half[i]), threads=1)
        assert l3[0] == 255 and bound[hard[i]] <= lo3[0] <= exact[hard[i]] and n3[0] == half[i]
    # max_length below the distance: unproven, and the lower bound exceeds max_length
    far = np.flatnonzero(exact >= 1)
    for cut in (0, 3, 7):
        sel = far[exact[far] > cut]
        a4, l4, lo4, _ = emul_solve(emul, tables, rows[sel], cut, 1 << 40)
        assert a4.shape == (len(sel), cut) and (a4 == 12).all()
        assert (l4 == 255).all() and (lo4 > cut).all() and (lo4 <= exact[sel] + 1).all()
    # unreachable rows: 255 everywhere, no node generated
    bad = np.concatenate(garbage(5, 20))
    b5, p5 = emul_bound(emul, tables, bad)
    a5, l5, lo5, n5 = emul_solve(emul, tables, bad, 14, 1 << 40)
    assert (b5 == 255).all() and (p5 == 255).all() and (l5 == 255).all() and (lo5 == 255).all()
    assert (a5 == 12).all() and (n5 == 0).all()


# ---- C ABI argument checks (no kernel is launched) -----------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    import rubiks_cube_solver_b200 as R
    from rubiks_cube_solver_b200 import _lib
    R.build_library()
    return _lib.load()


def test_pattern_argument_errors_without_cuda(lib):
    from rubiks_cube_solver_b200 import _lib
    buf = (ctypes.c_uint8 * 256)()
    base = ctypes.addressof(buf)
    al = ctypes.c_void_p((base + 15) & ~15)
    odd = ctypes.c_void_p(((base + 15) & ~15) + 4)
    assert lib.cube_pattern_tables_bytes(3) == 173335680
    assert lib.cube_pattern_tables_bytes(2) == _lib.CUBE_ERR_SIZE and b"cube_size 3" in lib.cube_last_error()
    assert lib.cube_pattern_tables_bytes(4) == _lib.CUBE_ERR_SIZE
    assert lib.cube_pattern_tables_build(2, al, None) == _lib.CUBE_ERR_SIZE
    assert lib.cube_distance_bound(2, al, al, 1, al, None, None) == _lib.CUBE_ERR_SIZE
    assert lib.cube_solve_bounded(2, al, al, 1, 14, 100, al, al, al, None, None) == _lib.CUBE_ERR_SIZE
    assert lib.cube_pattern_tables_build(3, None, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_distance_bound(3, None, al, 1, al, None, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_distance_bound(3, al, None, 1, al, None, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_distance_bound(3, al, al, -1, al, None, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_distance_bound(3, al, al, 1, None, None, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_solve_bounded(3, None, al, 1, 14, 100, al, al, al, None, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_solve_bounded(3, al, None, 1, 14, 100, al, al, al, None, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_solve_bounded(3, al, al, -1, 14, 100, al, al, al, None, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_solve_bounded(3, al, al, 1, -1, 100, al, al, al, None, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_solve_bounded(3, al, al, 1, 21, 100, al, al, al, None, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_solve_bounded(3, al, al, 1, 14, -1, al, al, al, None, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_solve_bounded(3, al, al, 1, 14, 100, al, None, al, None, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_pattern_tables_build(3, odd, None) == _lib.CUBE_ERR_ALIGN
    assert lib.cube_distance_bound(3, odd, al, 1, al, None, None) == _lib.CUBE_ERR_ALIGN
    assert lib.cube_distance_bound(3, al, odd, 1, al, None, None) == _lib.CUBE_ERR_ALIGN          # a misaligned row
    assert lib.cube_solve_bounded(3, al, odd, 1, 14, 100, al, al, al, None, None) == _lib.CUBE_ERR_ALIGN
    assert lib.cube_solve_bounded(3, al, al, 1, 14, 100, al, al, al, odd, None) == _lib.CUBE_ERR_ALIGN
    assert lib.cube_distance_bound(3, al, al, 0, None, None, None) == 0                    # nothing to do
    from rubiks_cube_solver_b200 import ops
    with pytest.raises(NotImplementedError):
        ops._pattern_bytes(2)
