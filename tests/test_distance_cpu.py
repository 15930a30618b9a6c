"""The exact 2x2x2 distance table without a GPU: the oracle's breadth-first search against the published
quarter-turn distribution, the table's invariants, the oracle's optimal solver, the reference checkpoint's
episodes against optimal, the per-state code of the distance kernels (csrc/cube_distance.cuh compiled with g++
by tests/host_emul/distance_emul.cpp) against the oracle, and the C ABI's argument checks."""
import ctypes
import hashlib
import os
import subprocess

import numpy as np
import pytest

from oracle import cube_np as O
from oracle import distance_np as D
from oracle import tables as T

HERE = os.path.dirname(os.path.abspath(__file__))

# states per distance 0..14 of the 2x2x2 in the quarter-turn metric, and the table's digest (rank order)
LEVELS = [1, 6, 27, 120, 534, 2256, 8969, 33058, 114149, 360508, 930588, 1350852, 782536, 90280, 276]
SHA256 = "de0634732a9d7224ed4525a24b857253201699fc5a8ac438989403c2da486f04"


@pytest.fixture(scope="session")
def table():
    return D.distance_table_2()


def _scrambles(n, seed, max_depth=40):
    rng = np.random.RandomState(seed)
    moves = rng.randint(6, size=(n, max_depth)).astype(np.uint8)
    moves[np.arange(max_depth)[None, :] >= rng.randint(0, max_depth + 1, size=(n, 1))] = 12   # depths 0..40
    out = np.empty((n, 24), dtype=np.uint8)
    for d in np.unique((moves < 6).sum(axis=1)):
        sel = (moves < 6).sum(axis=1) == d
        out[sel] = O.scramble(2, moves[sel, :d])
    return out


def _garbage(seed):
    """Rows that are no reachable state: random bytes, colours >= 6, two stickers swapped, a twisted corner."""
    rng = np.random.RandomState(seed)
    good = _scrambles(400, seed + 1)
    rnd = rng.randint(0, 256, size=(100, 24)).astype(np.uint8)
    colour = good[:100].copy()
    colour[np.arange(100), rng.randint(24, size=100)] = rng.randint(6, 256, size=100)
    swapped = good[100:200].copy()
    for row in swapped:                                       # two stickers of different colours exchanged
        i, j = rng.choice(24, size=2, replace=False)
        while row[i] == row[j]:
            i, j = rng.choice(24, size=2, replace=False)
        row[i], row[j] = row[j], row[i]
    twisted = good[200:300].copy()
    slots = T.PIECE_DEFS_2[rng.randint(7, size=100)]
    twisted[np.arange(100)[:, None], slots] = twisted[np.arange(100)[:, None], np.roll(slots, 1, axis=1)]
    return np.concatenate([rnd, colour, swapped, twisted])


def test_oracle_table_is_the_published_distribution(table):
    assert np.bincount(table, minlength=256)[:15].tolist() == LEVELS
    assert (table != D.UNREACHABLE).all() and len(table) == D.DISTANCE_ENTRIES_2 == 3674160
    assert hashlib.sha256(table.tobytes()).hexdigest() == SHA256
    assert table[0] == 0 and D.rank_2(O.solved_states(2, 1))[0] == 0


def test_every_state_has_a_closer_child_and_all_children_are_one_level_away(table):
    """A quarter turn is an odd permutation of the corners, so neighbours differ by exactly one level."""
    for lo in range(0, D.DISTANCE_ENTRIES_2, 1 << 19):
        ranks = np.arange(lo, min(lo + (1 << 19), D.DISTANCE_ENTRIES_2))
        states = D.unrank_2(ranks)
        d = table[ranks].astype(np.int64)
        kid_d = np.stack([table[D._rank_of_op(*np.moveaxis(O.get_op(2, O.apply_moves(2, states, np.full(len(ranks), a))), 2, 0))]
                          for a in range(6)], axis=1).astype(np.int64)
        assert (np.abs(kid_d - d[:, None]) == 1).all()
        assert ((kid_d == d[:, None] - 1).any(axis=1) | (d == 0)).all()


def test_rank_round_trip_and_unreachable_rows():
    ranks = np.random.RandomState(0).randint(0, D.DISTANCE_ENTRIES_2, size=20000)
    assert (D.rank_2(D.unrank_2(ranks)) == ranks).all()
    assert (D.rank_2(_scrambles(5000, 1)) >= 0).all()
    assert (D.rank_2(_garbage(2)) == -1).all()


def test_oracle_optimal_solutions(table):
    states = _scrambles(3000, 3)
    actions, length = D.solve_optimal_2(table, states)
    assert (length == D.distance_2(table, states)).all()
    assert ((actions < 6).sum(axis=1) == length).all() and (actions[length == 0] == 12).all()
    for k in range(14):                                       # the NOOP padding comes after the solution
        assert ((actions[:, k] < 6) == (k < length)).all()
    end = states.copy()
    for k in range(14):
        live = actions[:, k] < 6
        end[live] = O.apply_moves(2, end[live], actions[live, k])
    assert O.is_solved(2, end).all()
    bad_actions, bad_length = D.solve_optimal_2(table, _garbage(4))
    assert (bad_length == 255).all() and (bad_actions == 12).all()


def test_reference_checkpoint_episodes_are_never_shorter_than_optimal(table):
    g = np.load(os.path.join(HERE, "golden", "pin222.npz"))
    starts = np.stack([O.scramble(2, np.random.RandomState(int(s)).randint(6, size=(1, int(d))))[0]
                       for d in g["depths"] for s in g["seeds"]])
    dist = D.distance_2(table, starts).reshape(g["solved_plain"].shape).astype(np.int64)
    for tag in ("plain", "mask"):
        solved, steps = g["solved_" + tag], g["steps_" + tag]
        assert (steps[solved] >= dist[solved]).all()
        assert (steps[solved & (dist > 0)] - dist[solved & (dist > 0)]).min() == 0      # some greedy solutions are optimal
    roots = np.stack([O.scramble(2, np.random.RandomState(int(s)).randint(6, size=(1, int(d))))[0] for s, d in g["mcts_cases"]])
    n_act = (g["mcts_actions"] >= 0).sum(axis=1)
    solved = g["mcts_solved"]
    assert (n_act[solved] >= D.distance_2(table, roots)[solved]).all()


# ---- the distance kernels' per-state code on the CPU ----------------------------------------------------
@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    lib_path = str(tmp_path_factory.mktemp("distance_emul") / "libdistance_emul.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-w", "-o", lib_path,
                           os.path.join(HERE, "host_emul", "distance_emul.cpp")])
    lib = ctypes.CDLL(lib_path)
    vp, ll = ctypes.c_void_p, ctypes.c_longlong
    lib.emul_dist2_entries.restype = ll
    lib.emul_dist2_roundtrip_failures.restype = ll
    lib.emul_dist2_rank.argtypes = [vp, ll, vp]
    lib.emul_dist2_build.argtypes = [vp]
    lib.emul_dist2_lookup.argtypes = [vp, vp, ll, vp]
    lib.emul_dist2_solve.argtypes = [vp, vp, ll, vp, vp]
    return lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def test_emulated_rank_unrank(emul):
    assert emul.emul_dist2_entries() == D.DISTANCE_ENTRIES_2
    assert emul.emul_dist2_roundtrip_failures() == 0           # unrank then rank: identity on every rank
    for rows in (_scrambles(100000, 5), D.unrank_2(np.random.RandomState(6).randint(0, D.DISTANCE_ENTRIES_2, 20000)),
                 _garbage(7)):
        rows = np.ascontiguousarray(rows)
        got = np.empty(len(rows), dtype=np.int64)
        emul.emul_dist2_rank(_p(rows), len(rows), _p(got))
        assert (got == D.rank_2(rows)).all()


def test_emulated_table_build_lookup_and_solve(emul, table):
    built = np.empty(D.DISTANCE_ENTRIES_2, dtype=np.uint8)
    emul.emul_dist2_build(_p(built))
    assert hashlib.sha256(built.tobytes()).hexdigest() == SHA256
    rows = np.ascontiguousarray(np.concatenate([_scrambles(20000, 8), _garbage(9)]))
    dist = np.empty(len(rows), dtype=np.uint8)
    emul.emul_dist2_lookup(_p(table), _p(rows), len(rows), _p(dist))
    assert (dist == D.distance_2(table, rows)).all()
    actions = np.empty((len(rows), 14), dtype=np.uint8)
    length = np.empty(len(rows), dtype=np.uint8)
    emul.emul_dist2_solve(_p(table), _p(rows), len(rows), _p(actions), _p(length))
    want_a, want_l = D.solve_optimal_2(table, rows)
    assert (actions == want_a).all() and (length == want_l).all()


# ---- C ABI argument checks (no kernel is launched) -----------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    import rubiks_cube_solver_b200 as R
    from rubiks_cube_solver_b200 import _lib
    R.build_library()
    return _lib.load()


def test_distance_argument_errors_without_cuda(lib):
    from rubiks_cube_solver_b200 import _lib
    buf = (ctypes.c_uint8 * 256)()
    base = ctypes.addressof(buf)
    aligned = ctypes.c_void_p((base + 15) & ~15)
    odd = ctypes.c_void_p(((base + 15) & ~15) + 8)
    assert lib.cube_distance_table_entries(2) == 3674160
    assert lib.cube_distance_table_entries(3) == _lib.CUBE_ERR_SIZE and b"cube_size 2" in lib.cube_last_error()
    assert lib.cube_distance_table_build(3, aligned, None) == _lib.CUBE_ERR_SIZE
    assert lib.cube_distance(3, aligned, aligned, 1, aligned, None) == _lib.CUBE_ERR_SIZE
    assert lib.cube_solve_optimal(3, aligned, aligned, 1, aligned, aligned, None) == _lib.CUBE_ERR_SIZE
    assert lib.cube_distance_table_build(2, None, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_distance(2, None, aligned, 1, aligned, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_distance(2, aligned, None, 1, aligned, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_distance(2, aligned, aligned, -1, aligned, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_solve_optimal(2, None, aligned, 1, aligned, aligned, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_solve_optimal(2, aligned, aligned, -1, aligned, aligned, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_distance_table_build(2, odd, None) == _lib.CUBE_ERR_ALIGN
    assert lib.cube_distance(2, aligned, odd, 1, aligned, None) == _lib.CUBE_ERR_ALIGN              # a misaligned row
    assert lib.cube_distance(2, odd, aligned, 1, aligned, None) == _lib.CUBE_ERR_ALIGN
    assert lib.cube_solve_optimal(2, aligned, odd, 1, aligned, aligned, None) == _lib.CUBE_ERR_ALIGN
    with pytest.raises(NotImplementedError):
        from rubiks_cube_solver_b200 import ops
        ops._distance_entries(3)
