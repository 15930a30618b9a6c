"""CPU emulation of the CUDA kernels' per-thread code (tests/host_emul/emul.cpp compiles
csrc/cube_threads.cuh as plain C++) against the oracle.  Catches table / selector / index
bugs without a GPU; the product library never contains this code path."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from oracle import cube_np as O
from oracle import tables as T

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "host_emul", "emul.cpp")
LIB = os.path.join(HERE, "host_emul", "libcube_emul.so")
CSRC = os.path.join(os.path.dirname(HERE), "rubiks_cube_solver_b200", "csrc")


@pytest.fixture(scope="module")
def emul():
    deps = [SRC] + [os.path.join(CSRC, f) for f in ("cube_threads.cuh", "cube_common.cuh", "cube_tables.cuh")]
    if not os.path.exists(LIB) or any(os.path.getmtime(d) > os.path.getmtime(LIB) for d in deps):
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-w", "-o", LIB, SRC])
    lib = ctypes.CDLL(LIB)
    vp, ll = ctypes.c_void_p, ctypes.c_longlong
    lib.emul_scramble.argtypes = [ctypes.c_int, vp, ll, ctypes.c_int, vp, vp]
    lib.emul_scramble_pairs.argtypes = [ctypes.c_int, vp, ll, ctypes.c_int, vp, vp, ctypes.c_int]
    lib.emul_scramble_step_pairs.argtypes = [ctypes.c_int, vp, vp, ll, ctypes.c_int, vp, vp, ctypes.c_int]
    lib.emul_scramble_sliced.argtypes = [ctypes.c_int, vp, vp, ll, ctypes.c_int, vp, vp, ctypes.c_int]
    lib.emul_prefixes.argtypes = [ctypes.c_int, vp, ll, ctypes.c_int, vp, vp]
    lib.emul_walk_private.argtypes = [ctypes.c_int, vp, vp, ll, ctypes.c_int, vp, vp]
    lib.emul_walk.argtypes = [ctypes.c_int, vp, vp, ll, ctypes.c_int, vp, vp]
    lib.emul_expand.argtypes = [ctypes.c_int, ctypes.c_int, vp, ll, vp, vp, vp, vp]
    return lib


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


@pytest.mark.parametrize("size", (2, 3))
@pytest.mark.parametrize("depth", (0, 1, 3, 4, 7, 8, 9, 20, 30, 31, 32, 61, 100))
def test_scramble_emulation(emul, size, depth):
    rng = np.random.RandomState(depth * 7 + size)
    n = 700                                   # two full tiles + a ragged one
    A = T.N_ACTIONS[size]
    moves = rng.randint(A, size=(n, depth)).astype(np.uint8)
    if depth >= 2:
        h = depth // 2
        moves[:50, h:2 * h] = moves[:50, :h][:, ::-1] ^ 1          # rows that come back to solved
        if depth % 2:
            moves[:50, -1] = moves[:50, 0]
    out = np.empty((n, T.N_STICKERS[size]), dtype=np.uint8)
    solved = np.empty(n, dtype=np.uint8)
    emul.emul_scramble(size, _p(moves), n, depth, _p(out), _p(solved))
    want = O.scramble(size, moves)
    assert (out == want).all()
    assert (solved.astype(bool) == O.is_solved(size, want)).all()
    if depth >= 2 and depth % 2 == 0:
        assert solved[:50].all()


@pytest.mark.parametrize("size", (2, 3))
@pytest.mark.parametrize("depth,fixed", [(d, 0) for d in (1, 2, 3, 4, 5, 7, 8, 9, 20, 30, 31, 32, 43, 61, 96, 100, 201, 318)]
                         + [(20, 1), (30, 1), (43, 1)]
                         + [(d, 2) for d in (8, 16, 24, 32, 48, 64, 72, 96, 128, 200, 320)]
                         + [(d, 4) for d in (1, 2, 3, 5, 8, 9, 10, 14, 19, 21, 30, 31)] + [(20, 5), (30, 5), (16, 6), (32, 6)])
def test_scramble_pairs_emulation(emul, size, depth, fixed):
    """K1p (two moves per table row, persistent 64-row tiles): rows that return to solved, the
    no-move index 12 in the stream, odd depths (padded tail pair) and the fold schedule.
    fixed & 3 = 2: the swizzled move tile the kernel uses where the flat image bank-conflicts;
    fixed & 4: four instances per lane (2x2x2, 128-row tiles)."""
    if fixed & 3 == 2 and size == 2 and depth % 16:
        pytest.skip("2x2x2 uses the swizzled tile for multiples of 16 only")
    if fixed & 4 and size == 3:
        pytest.skip("four instances per lane: 2x2x2 only")
    rng = np.random.RandomState(depth * 11 + size)
    n = 384 if fixed & 4 else 192
    A = T.N_ACTIONS[size]
    moves = rng.randint(A, size=(n, depth)).astype(np.uint8)
    if depth >= 2:
        h = depth // 2
        moves[:50, h:2 * h] = moves[:50, :h][:, ::-1] ^ 1          # rows that come back to solved
        if depth % 2:
            moves[:50, -1] = 12
    moves[60:90][rng.rand(30, depth) < 0.3] = 12                     # no-move index anywhere
    if size == 2:                                                    # 2x2x2: every index A..12 is a no-op
        sub = moves[90:120]
        sub[rng.rand(30, depth) < 0.3] = rng.randint(6, 13)
    out = np.empty((n, T.N_STICKERS[size]), dtype=np.uint8)
    solved = np.empty(n, dtype=np.uint8)
    emul.emul_scramble_pairs(size, _p(moves), n, depth, _p(out), _p(solved), fixed)
    want = np.empty_like(out)
    for i in range(n):                                               # the oracle skips the no-move indices
        row = moves[i][moves[i] < A]
        want[i] = O.scramble(size, row[None, :])[0]
    assert (out == want).all()
    assert (solved.astype(bool) == O.is_solved(size, want)).all()
    if depth >= 2:
        assert solved[:50].all()


@pytest.mark.parametrize("size", (2, 3))
def test_pair_twist_field_never_overflows(size):
    """K1p adds the composed twist of two moves (0..2 per corner) to a 5-bit field: no fold for
    depth <= 30 (15 pairs), a fold every 10 pairs beyond.  Worst case of that schedule, exactly."""
    worst, f = 0, 0
    for pair in range(1, 16):
        f += 2
        worst = max(worst, f)
    assert worst <= 31                                              # depth <= 30, never folded
    f, worst, after = 0, 0, 0
    for word in range(1, 400):                                      # generic path: fold after every 5th word
        f += 4
        worst = max(worst, f)
        if word % 5 == 0:
            f = after = max(after, max((v & 3) + (v >> 2) for v in range(f + 1)))
    assert worst <= 31 and after + 4 * 4 + 4 <= 31                  # <= 4 left-over words and the tail word


@pytest.mark.parametrize("size", (2, 3))
def test_scramble_emulation_noop_rows(emul, size):
    # indices A..15 are no-ops on the hot path (include/cube_b200.h)
    rng = np.random.RandomState(3)
    A = T.N_ACTIONS[size]
    moves = rng.randint(A, size=(300, 12)).astype(np.uint8)
    padded = np.full((300, 24), 12, dtype=np.uint8)
    padded[:, ::2] = moves
    a = np.empty((300, T.N_STICKERS[size]), dtype=np.uint8)
    s = np.empty(300, dtype=np.uint8)
    emul.emul_scramble(size, _p(padded), 300, 24, _p(a), _p(s))
    assert (a == O.scramble(size, moves)).all()


@pytest.mark.parametrize("size", (2, 3))
@pytest.mark.parametrize("depth", (1, 5))
def test_walk_emulation(emul, size, depth):
    rng = np.random.RandomState(11 + size)
    n = 600
    A = T.N_ACTIONS[size]
    start = O.scramble(size, rng.randint(A, size=(n, 9)))
    start[:20] = rng.randint(0, 256, size=(20, T.N_STICKERS[size]))     # arbitrary bytes: still a pure gather
    moves = rng.randint(A, size=(n, depth)).astype(np.uint8)
    start[20:40] = O.scramble(size, (moves[20:40, ::-1] ^ 1))           # rows that end solved
    out = np.empty_like(start)
    solved = np.empty(n, dtype=np.uint8)
    emul.emul_walk(size, _p(start), _p(moves), n, depth, _p(out), _p(solved))
    want = O.scramble(size, moves, init=start)
    assert (out == want).all()
    assert (solved.astype(bool) == O.is_solved(size, want)).all()
    assert solved[20:40].all()


@pytest.mark.parametrize("size", (2, 3))
@pytest.mark.parametrize("depth", (1, 2, 5))
def test_walk_private_emulation(emul, size, depth):
    """K2p (lane-private scratch layout, 64-row tiles, even / odd row passes): arbitrary bytes stay a
    pure gather, rows that end solved are flagged, neighbours' bytes survive the in-place write-back."""
    rng = np.random.RandomState(21 + size + depth)
    n = 192
    A = T.N_ACTIONS[size]
    start = O.scramble(size, rng.randint(A, size=(n, 9)))
    start[:20] = rng.randint(0, 256, size=(20, T.N_STICKERS[size]))
    moves = rng.randint(A, size=(n, depth)).astype(np.uint8)
    moves[40:60, -1] = 12                                                # no-op row
    start[20:40] = O.scramble(size, (moves[20:40, ::-1] ^ 1))           # rows that end solved
    out = np.empty_like(start)
    solved = np.empty(n, dtype=np.uint8)
    emul.emul_walk_private(size, _p(start), _p(moves), n, depth, _p(out), _p(solved))
    want = start.copy()
    for i in range(n):
        row = moves[i][moves[i] < A]
        want[i] = O.scramble(size, row[None, :], init=start[i:i + 1])[0]
    assert (out == want).all()
    assert (solved.astype(bool) == O.is_solved(size, want)).all()
    assert solved[20:40].all()


@pytest.mark.parametrize("size", (2, 3))
@pytest.mark.parametrize("dtype", (0, 1, 2))
@pytest.mark.parametrize("n", (5, 16, 37))
def test_expand_emulation(emul, size, dtype, n):
    rng = np.random.RandomState(n + dtype)
    A, S = T.N_ACTIONS[size], T.N_STICKERS[size]
    D = T.ONEHOT_WIDTH[size]
    parents = O.scramble(size, rng.randint(A, size=(n, 6)))
    parents[0] = O.scramble(size, np.array([[3]]))[0]                    # one move from solved
    es = (2, 4, 1)[dtype]
    children = np.empty((n, A, S), dtype=np.uint8)
    coh = np.empty((n, A, D * es), dtype=np.uint8)
    poh = np.empty((n, D * es), dtype=np.uint8)
    solved = np.empty((n, A), dtype=np.uint8)
    emul.emul_expand(size, dtype, _p(parents), n, _p(children), _p(coh), _p(poh), _p(solved))
    want_c, want_s = O.expand(size, parents)
    assert (children == want_c).all() and (solved.astype(bool) == want_s).all()
    assert solved[0, 2] == 1
    one = {0: np.uint16(0x3f80), 1: np.float32(1.0), 2: np.uint8(1)}[dtype]
    view = {0: np.uint16, 1: np.float32, 2: np.uint8}[dtype]
    want_coh = O.encode(size, want_c.reshape(n * A, S)).reshape(n, A, D).astype(view) * one
    want_poh = O.encode(size, parents).reshape(n, D).astype(view) * one
    assert (coh.view(view).reshape(n, A, D) == want_coh).all()
    assert (poh.view(view).reshape(n, D) == want_poh).all()


def twin_rows(size, n, seed):
    """Sticker rows the reference encodes but no turn sequence reaches: a random scramble in which one cubie's
    stickers are copied onto another cubie position -- as they are, or turned (3x3x3 edges also flipped) -- so the
    row names one piece twice and leaves another out.  Only rows the reference's table lookup accepts are kept
    (O.encode raises IndexError on a hash outside its table)."""
    rng = np.random.RandomState(seed)
    A = T.N_ACTIONS[size]
    rows = []
    while len(rows) < n:
        row = O.scramble(size, rng.randint(A, size=(1, 9)))[0]
        groups = [T.PIECE_DEFS_2] if size == 2 else [T.CORNER_DEFS_3, T.EDGE_DEFS_3]
        defs = groups[rng.randint(len(groups))]
        src, dst = rng.choice(len(defs), 2, replace=False)
        row[defs[dst]] = np.roll(row[defs[src]], rng.randint(defs.shape[1]))
        try:
            O.encode(size, row[None])
        except IndexError:
            continue
        rows.append(row)
    return np.stack(rows)


def _expand_emulation_vs_oracle(emul, size, dtype, parents):
    n = parents.shape[0]
    A, S, D = T.N_ACTIONS[size], T.N_STICKERS[size], T.ONEHOT_WIDTH[size]
    es = (2, 4, 1)[dtype]
    children = np.empty((n, A, S), dtype=np.uint8)
    coh = np.empty((n, A, D * es), dtype=np.uint8)
    poh = np.empty((n, D * es), dtype=np.uint8)
    solved = np.empty((n, A), dtype=np.uint8)
    emul.emul_expand(size, dtype, _p(parents), n, _p(children), _p(coh), _p(poh), _p(solved))
    want_c, want_s = O.expand(size, parents)
    assert (children == want_c).all() and (solved.astype(bool) == want_s).all()
    one = {0: np.uint16(0x3f80), 1: np.float32(1.0), 2: np.uint8(1)}[dtype]
    view = {0: np.uint16, 1: np.float32, 2: np.uint8}[dtype]
    want_coh = O.encode(size, want_c.reshape(n * A, S)).reshape(n, A, D).astype(view) * one
    want_poh = O.encode(size, parents).reshape(n, D).astype(view) * one
    assert (coh.view(view).reshape(n, A, D) == want_coh).all()
    assert (poh.view(view).reshape(n, D) == want_poh).all()


@pytest.mark.parametrize("size", (2, 3))
@pytest.mark.parametrize("dtype", (0, 1, 2))
@pytest.mark.parametrize("n", (5, 37, 64, 128))
def test_expand_emulation_rows_that_name_a_piece_twice(emul, size, dtype, n):
    """Rows that name a cubie twice among reachable rows, in whole and ragged tiles.  2x2x2: the reference's loop
    (cube_env.py:141-147) sets one 1 per position, so the twice-named cubelet's one-hot row has two 1s and the
    missing cubelet's none -- a tile with such a row takes the element-wise path.  3x3x3 writes one column per
    slot and is unaffected; this pins it."""
    rng = np.random.RandomState(100 * size + n + dtype)
    parents = O.scramble(size, rng.randint(T.N_ACTIONS[size], size=(n, 6)))
    at = sorted({0, n // 2, n - 1})
    parents[at] = twin_rows(size, len(at), seed=n + dtype)
    if size == 2:
        assert (O.encode(2, parents[at]).sum(axis=2) == 2).any(axis=1).all()        # the case under test
    _expand_emulation_vs_oracle(emul, size, dtype, parents)


_ARBITRARY_BYTES_SCRIPT = r"""
import ctypes, sys
import numpy as np
sys.path.insert(0, sys.argv[2])
from oracle import tables as T
lib = ctypes.CDLL(sys.argv[1])
vp, ll = ctypes.c_void_p, ctypes.c_longlong
lib.emul_expand.argtypes = [ctypes.c_int, ctypes.c_int, vp, ll, vp, vp, vp, vp]
p = lambda a: a.ctypes.data_as(vp)
rng = np.random.RandomState(5)
for size in (2, 3):
    A, S, D = T.N_ACTIONS[size], T.N_STICKERS[size], T.ONEHOT_WIDTH[size]
    for dtype, es, one in ((0, 2, 0x3f80), (1, 4, 0x3f800000), (2, 1, 1)):
        for n in (37, 64, 129):
            parents = rng.randint(0, 256, size=(n, S)).astype(np.uint8)
            parents[::3] = rng.randint(0, 8, size=parents[::3].shape)
            children = np.empty((n, A, S), dtype=np.uint8)
            coh = np.empty((n, A, D * es), dtype=np.uint8)
            poh = np.empty((n, D * es), dtype=np.uint8)
            solved = np.empty((n, A), dtype=np.uint8)
            lib.emul_expand(size, dtype, p(parents), n, p(children), p(coh), p(poh), p(solved))
            assert (children == parents[:, T.MOVE_DEFS[size]]).all()
            assert set(np.unique(solved)) <= {0, 1}
            view = {0: np.uint16, 1: np.uint32, 2: np.uint8}[dtype]
            for oh in (coh, poh):
                assert set(np.unique(oh.view(view))) <= {0, one}, (size, dtype, n)
print("ok")
"""


def test_expand_emulation_arbitrary_bytes_under_address_sanitizer(tmp_path):
    """Colour bytes >= 6 (and any other byte) are outside the reference's domain but must stay memory-safe: every
    table index is masked.  The emulation built with AddressSanitizer and libstdc++ assertions runs such rows
    through every size and dtype, in whole and ragged tiles: no out-of-range access, one-hot elements 0 or 1,
    flags 0 or 1, children still the plain gather."""
    lib = str(tmp_path / "libcube_emul_asan.so")
    rt = subprocess.run(["g++", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not os.path.isabs(rt) or not os.path.exists(rt):
        pytest.skip("g++ has no AddressSanitizer runtime")
    subprocess.check_call(["g++", "-O1", "-g", "-std=c++17", "-shared", "-fPIC", "-w", "-fsanitize=address",
                           "-fno-omit-frame-pointer", "-D_GLIBCXX_ASSERTIONS", "-o", lib, SRC])
    env = dict(os.environ, LD_PRELOAD=rt, ASAN_OPTIONS="detect_leaks=0:abort_on_error=0")
    out = subprocess.run([sys.executable, "-c", _ARBITRARY_BYTES_SCRIPT, lib, os.path.dirname(HERE)], capture_output=True,
                         text=True, timeout=300, env=env)
    assert out.returncode == 0 and out.stdout.strip().endswith("ok"), out.stdout[-2000:] + out.stderr[-4000:]


def _gen_tables():
    import importlib.util
    spec = importlib.util.spec_from_file_location("_gen_t", os.path.join(CSRC, "gen_tables.py"))
    g = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(g)
    return g


@pytest.mark.parametrize("size", (2, 3))
def test_lazy_twist_field_never_overflows(size):
    """The scramble kernel accumulates corner twists un-reduced in a 5-bit field and folds it
    every 4 turns.  Exact integer model of that schedule: random walks plus a greedy adversary
    that always plays the turn maximising the largest field must stay below 32."""
    g = _gen_tables()
    src, rot = (g.C_SRC_3, g.C_ROT_3) if size == 3 else (g.C_SRC_2, g.C_ROT_2)
    n_moves = len(src)

    def gain(m, q):                         # c0 += B, c1 += 2*B (cube_common.cuh cubie_move_at)
        return int(rot[m][q]) if q < 4 else 2 * int(rot[m][q - 4])

    def turn(field, m):
        return [field[src[m][q]] + gain(m, q) for q in range(8)]

    def fold(field):
        return [(f & 3) + (f >> 2) for f in field]

    rng = np.random.RandomState(0)
    worst = 0
    for trial in range(400):
        field = [0] * 8
        for k in range(64):
            if trial < 200:
                m = int(rng.randint(n_moves))
            else:                            # greedy adversary with random tie-breaks
                cands = [(max(turn(field, mm)), rng.rand(), mm) for mm in range(n_moves)]
                m = max(cands)[2]
            field = turn(field, m)
            worst = max(worst, max(field))
            assert max(field) < 32, (trial, k, field)
            if k % 4 == 3:
                field = fold(field)
                assert max(field) <= 8
    assert worst <= 24


@pytest.mark.parametrize("size", (2, 3))
@pytest.mark.parametrize("depth", (1, 2, 3, 4, 5, 8, 29, 30, 31, 64, 131))
def test_prefixes_emulation(emul, size, depth):
    """K1x (cube_scramble_prefixes): the per-lane walk of prefix.cu -- lazy twist folds every four moves, every
    level finished on a copy into the tile image at row lane * depth + k (rows of both parities) -- against the
    oracle's per-step states and done flags; a ragged last tile."""
    rng = np.random.RandomState(depth + 50 * size)
    n = 32 * 3 + 7
    A = T.N_ACTIONS[size]
    moves = rng.randint(A, size=(n, depth)).astype(np.uint8)
    if depth >= 4:
        moves[::2, 2:4] = moves[::2, :2][:, ::-1] ^ 1
    out = np.empty((n, depth, T.N_STICKERS[size]), dtype=np.uint8)
    solved = np.empty((n, depth), dtype=np.uint8)
    emul.emul_prefixes(size, _p(moves), n, depth, _p(out), _p(solved))
    _, want, flags = O.scramble(size, moves, per_step=True)
    assert (out == want).all() and (solved.astype(bool) == flags).all()
    if depth >= 4:
        assert solved[0, 3] == 1


@pytest.mark.parametrize("size", (2, 3))
@pytest.mark.parametrize("depth,fixed", [(d, 0) for d in (1, 2, 7, 29, 31, 100, 319)] + [(30, 1), (20, 1), (32, 2), (96, 2), (320, 2)]
                         + [(20, 5), (30, 5), (9, 4)])
def test_scramble_step_pairs_emulation(emul, size, depth, fixed):
    """cube_scramble_step through K1p: the walk of `depth` moves leaves twist fields as large as 30; the trailing
    action (fold, then the pair row (action, no move)) must still give the depth + 1 scramble of the oracle."""
    if (fixed & 4) and size == 3:
        pytest.skip("four instances per lane is a 2x2x2 variant")
    if (fixed & 3) == 2 and depth % (8 if size == 3 else 16):
        pytest.skip("swizzled tiles need depth % 8 (3x3x3) / % 16 (2x2x2) == 0")
    rng = np.random.RandomState(3 * depth + size + fixed)
    tile = 128 if fixed & 4 else 64
    n = tile * 3
    A = T.N_ACTIONS[size]
    moves = rng.randint(A, size=(n, depth)).astype(np.uint8)
    if size == 3 and depth >= 2:
        moves[:32] = np.tile(np.array([2, 4], dtype=np.uint8), (32, depth // 2 + 1))[:, :depth]   # F R F R ...: twists pile up
    last = rng.randint(A, size=n).astype(np.uint8)
    last[::5] = 12                                                      # the no-move index as the action
    out = np.empty((n, T.N_STICKERS[size]), dtype=np.uint8)
    solved = np.empty(n, dtype=np.uint8)
    emul.emul_scramble_step_pairs(size, _p(moves), _p(last), n, depth, _p(out), _p(solved), fixed)
    want = O.scramble(size, moves)
    stepped = want.copy()
    real = last < A
    stepped[real] = O.apply_moves(size, want[real], last[real])
    assert (out == stepped).all()
    assert (solved.astype(bool) == O.is_solved(size, stepped)).all()


@pytest.mark.parametrize("size", (2, 3))
@pytest.mark.parametrize("slice_len", (112, 240))
@pytest.mark.parametrize("depth,with_last", [(321, 0), (400, 0), (479, 1), (480, 0), (481, 0), (482, 0), (483, 1), (495, 0), (723, 0), (1000, 1), (241, 0), (17, 0), (254, 0)])
def test_scramble_sliced_emulation(emul, size, depth, with_last, slice_len):
    """K1p sliced (deep scrambles): pieces staged from the 16-byte boundary below them into 272-byte slots (the
    host harness aborts on a misaligned 128-bit load), every per-row shift 0..15 taken out by the word select +
    funnel, slices that end in 1..15 left-over moves, the cubie state carried from slice to slice with a fold
    at every slice start and after every unit (worst case: F R F R ... piles the twists up) -- against the oracle."""
    rng = np.random.RandomState(depth + size)
    n = 64 * 2
    A = T.N_ACTIONS[size]
    moves = np.zeros(n * depth + 16, dtype=np.uint8)                    # readable 16 bytes past the end
    m2 = moves[:n * depth].reshape(n, depth)
    m2[:] = rng.randint(A, size=(n, depth))
    m2[:8] = np.tile(np.array([2, 4], dtype=np.uint8), (8, depth // 2 + 1))[:, :depth]
    h = depth // 2
    m2[8:24, h:2 * h] = m2[8:24, :h][:, ::-1] ^ 1                       # back to solved (then one more move if odd)
    last = rng.randint(A, size=n).astype(np.uint8) if with_last else None
    out = np.empty((n, T.N_STICKERS[size]), dtype=np.uint8)
    solved = np.empty(n, dtype=np.uint8)
    emul.emul_scramble_sliced(size, _p(moves), _p(last), n, depth, _p(out), _p(solved), slice_len)
    want = O.scramble(size, m2)
    if with_last:
        want = O.apply_moves(size, want, last)
    assert (out == want).all()
    assert (solved.astype(bool) == O.is_solved(size, want)).all()
    if depth % 2 == 0 and not with_last:
        assert solved[8:24].all()


def test_row_assembly_takes_the_centres_from_edge_lut_words():
    """K1p's finishing pass (gen_tables.py: E_LUT_SLOT_3, assemble_row_fn): every edge slot's LUT carries the centre
    colours of the slot's two faces in bytes 2 and 3, both alignments of the row assembly need 32 byte permutes
    (38 with the centres as immediates), and no centre immediate is left in the generated code."""
    g = _gen_tables()
    assert len(g.E_LUT_SLOT_3) == 12 and all(len(lut) == 32 for lut in g.E_LUT_SLOT_3)
    for slot, lut in zip(g.EDGE_SLOTS_3, g.E_LUT_SLOT_3):
        for i, v in enumerate(lut):
            assert v & 0xffff == g._E_LUT_32[i] & 0xffff                      # the two colours, as in the shared LUT
            assert (v >> 16) & 0xff == slot[0] // 9 and v >> 24 == slot[1] // 9
    for f in range(6):                                                        # four edge stickers per face
        assert len(g.CENTRE_ALTERNATIVES_3[f]) == 4
    src3 = g.sticker_sources([g.CORNER_SLOTS_3, g.EDGE_SLOTS_3], 54, {4 + 9 * f: f for f in range(6)})
    for first, half_at in ((0, 52), (2, 0)):
        with_alt = g.assemble_row_fn("f", src3, first, 13, half_at, g.CENTRE_ALTERNATIVES_3)
        without = g.assemble_row_fn("f", src3, first, 13, half_at)
        assert "// 32 byte permutes" in with_alt and "// 38 byte permutes" in without
        # no immediate operand (a centre constant) remains: operands are L[..] words and nested permutes only
        body = with_alt.split("{", 1)[1]
        assert not re.search(r"cube_prmt\((0x[0-9a-f]{2}u)|, (0x[0-9a-f]{2}u),", body)
