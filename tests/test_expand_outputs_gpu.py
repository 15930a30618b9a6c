"""The expansion family -- cube_expand, cube_expand_codes, cube_encode, cube_solved and cube_decode -- with every
set of optional outputs against the oracle.

launch_expand (csrc/expand.cu) picks a kernel from WHICH outputs the caller passed and the dtype: a 2x2x2 call
with the children's one-hot rows in bf16 / u8 runs K3c (leaf_children_kernel) on whole tiles of 16 parents and the
generic expand_kernel on the rest; in f32 the generic kernel takes every parent; with children or the parent's
one-hot rows but no child one-hot rows leaf_kernel takes whole tiles of 64 and the generic kernel (or, for the
parent's one-hot rows alone, encode_kernel) the rest; cube_expand_codes always runs the generic kernel; 3x3x3 runs
expand_kernel / encode_kernel with the reference or the exact encoding.  Every present output lives between guard
bytes and is compared bit for bit; the batch sizes put ragged tails behind whole tiles of every kernel.

Rows that name a 2x2x2 cubelet twice (no real state does, but the reference encodes them: cube_env.py:141-147
sets one 1 per position) are planted at both sides of tile boundaries and must get the reference's one-hot rows
from every kernel and front end.  Rows with colour bytes >= 6 are outside the reference's domain and must stay
memory-safe."""
import itertools
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import rubiks_cube_solver_b200 as R
from rubiks_cube_solver_b200 import _lib, ops

from oracle import cube_c as C
from oracle import cube_np as O
from oracle import tables as T
from test_host_emulation import twin_rows
from test_optional_outputs_gpu import Guarded, _counters, _kernel_key, _ptr, _stream, cu, dev

pytestmark = pytest.mark.gpu
SIZES = (2, 3)
DTYPE_IDS = ("bf16", "f32", "u8")
ESIZE = (2, 4, 1)
TORCH_DTYPE = (torch.bfloat16, torch.float32, torch.uint8)
ONE = (np.uint16(0x3f80), np.uint32(0x3f800000), np.uint8(1))       # the bits of 1 in each dtype
NP_BITS = (np.uint16, np.uint32, np.uint8)
OUTS = ("children", "child_onehot", "parent_onehot", "solved", "reward")
ONEHOT_OUTS = {"child_onehot", "parent_onehot"}
# 2x2x2: 40 leaf tiles + 37 (162 K3c tiles + 5); whole tiles only; fewer parents than a K3c tile.  3x3x3: 150 tiles
# of the generic kernel + 5, and one parent.
EXPAND_N = {2: (64 * 40 + 37, 64 * 8, 11), 3: (16 * 150 + 5, 1)}
TWIN_AT = (0, 63, 64, 65)                                       # and the last row: both sides of tile boundaries


def subsets(items):
    return [frozenset(c) for k in range(len(items) + 1) for c in itertools.combinations(items, k)]


def onehot_bits(size, states, dtype, exact):
    """The oracle's one-hot rows of `states` as the bytes the library writes in `dtype`."""
    enc = O.encode_exact(states) if (size == 3 and exact) else O.encode(size, states)
    return (enc.reshape(len(states), -1).astype(NP_BITS[dtype]) * ONE[dtype]).view(np.uint8).reshape(-1)


def codes_of(size, states, exact):
    """argmax over every oracle one-hot row, zero-padded to key_bytes (cube_expand_codes)."""
    enc = O.encode_exact(states) if (size == 3 and exact) else O.encode(size, states)
    codes = np.zeros((len(states), ops.key_bytes(size)), dtype=np.uint8)
    codes[:, :enc.shape[1]] = enc.argmax(axis=2)
    return codes


def parents_of(size, n, seed=0):
    """Scrambled parents, every seventh one move from solved (so it has a solved child)."""
    rng = np.random.RandomState(1000 * size + n + seed)
    A = T.N_ACTIONS[size]
    parents = C.scramble(size, rng.randint(A, size=(n, 8)).astype(np.uint8))[0]
    parents[::7] = C.scramble(size, rng.randint(A, size=((n + 6) // 7, 1)).astype(np.uint8))[0]
    return np.ascontiguousarray(parents)


def plant_twins(parents, seed=0):
    """The same 2x2x2 row that names a cubelet twice at indices 0, 63, 64, 65 and n - 1 (those that exist)."""
    n = len(parents)
    at = sorted({i for i in TWIN_AT if i < n} | {n - 1})
    parents[at] = twin_rows(2, 1, seed)[0]
    assert (O.encode(2, parents[at]).sum(axis=2) == 2).any(axis=1).all()
    return parents


class Want(object):
    """Everything the oracle says about one batch of parents."""

    def __init__(self, size, parents, exact):
        self.size, self.parents, self.exact, self.n = size, parents, exact, len(parents)
        A, S = T.N_ACTIONS[size], T.N_STICKERS[size]
        self.children = C.expand(size, parents, want_cols=False)[0]
        self.solved = O.is_solved(size, self.children.reshape(-1, S)).reshape(self.n, A)
        self.reward = np.where(self.solved, np.float32(1.0), np.float32(-1.0)).astype(np.float32)
        self._bits = {}

    def child_onehot(self, dtype):
        if ("c", dtype) not in self._bits:
            rows = self.children.reshape(self.n * T.N_ACTIONS[self.size], -1)
            self._bits["c", dtype] = onehot_bits(self.size, rows, dtype, self.exact)
        return self._bits["c", dtype]

    def parent_onehot(self, dtype):
        if ("p", dtype) not in self._bits:
            self._bits["p", dtype] = onehot_bits(self.size, self.parents, dtype, self.exact)
        return self._bits["p", dtype]

    def child_codes(self):
        return codes_of(self.size, self.children.reshape(self.n * T.N_ACTIONS[self.size], -1), self.exact).reshape(-1)

    def parent_codes(self):
        return codes_of(self.size, self.parents, self.exact).reshape(-1)


def host(g):
    return g.view.cpu().numpy()


def check_outputs(want, got, dtype, counters, what):
    for name, g in list(got.items()) + [("counters", counters)]:
        assert g is None or g.intact(), "%s: %s guard bytes overwritten" % (what, name)
    if "children" in got:
        assert (host(got["children"]) == want.children.reshape(-1)).all(), what
    if "solved" in got:
        assert (host(got["solved"]) == want.solved.reshape(-1).astype(np.uint8)).all(), what
    if "reward" in got:
        assert (host(got["reward"]).view(np.float32) == want.reward.reshape(-1)).all(), what
    if "child_onehot" in got:
        assert (host(got["child_onehot"]) == want.child_onehot(dtype)).all(), what
    if "parent_onehot" in got:
        assert (host(got["parent_onehot"]) == want.parent_onehot(dtype)).all(), what
    if "child_codes" in got:
        assert (host(got["child_codes"]) == want.child_codes()).all(), what
    if "parent_codes" in got:
        assert (host(got["parent_codes"]) == want.parent_codes()).all(), what
    if counters is not None:
        assert counters.view.tolist() == [int(want.solved.sum()), want.n * T.N_ACTIONS[want.size], 0, 0], what


def buffers(size, n, outs, dtype):
    A, S, D, K = T.N_ACTIONS[size], T.N_STICKERS[size], T.ONEHOT_WIDTH[size], ops.key_bytes(size)
    per = {"children": n * A * S, "child_onehot": n * A * D * ESIZE[dtype], "parent_onehot": n * D * ESIZE[dtype],
           "solved": n * A, "reward": 4 * n * A, "child_codes": n * A * K, "parent_codes": n * K}
    return {name: Guarded(per[name]) for name in outs}


def run_expand(size, states, outs, dtype, with_counters, encoding):
    """cube_expand with the outputs `outs`, each between guard bytes."""
    n = states.shape[0]
    got = buffers(size, n, outs, dtype)
    counters = _counters() if with_counters else None
    p = lambda name: _ptr(got[name].view) if name in got else None
    rc = _lib.load().cube_expand(size, _ptr(states), n, p("children"), p("child_onehot"), p("parent_onehot"), dtype,
                                 encoding, p("solved"), p("reward"), counters and _ptr(counters.view), _stream())
    _lib.check(rc, "cube_expand")
    torch.cuda.synchronize()
    return got, counters


def run_expand_codes(size, states, outs, dtype, with_counters, encoding):
    n = states.shape[0]
    got = buffers(size, n, outs, dtype)
    counters = _counters() if with_counters else None
    p = lambda name: _ptr(got[name].view) if name in got else None
    rc = _lib.load().cube_expand_codes(size, _ptr(states), n, p("children"), p("child_codes"), p("parent_codes"),
                                       p("parent_onehot"), dtype, encoding, p("solved"), p("reward"),
                                       counters and _ptr(counters.view), _stream())
    _lib.check(rc, "cube_expand_codes")
    torch.cuda.synchronize()
    return got, counters


# ------------------------------------------------------------------ cube_expand
EXPAND_CASES = [(2, 0, n) for n in EXPAND_N[2]] + [(2, 1, EXPAND_N[2][0])] + \
               [(3, e, n) for e in (0, 1) for n in EXPAND_N[3]]


@pytest.mark.parametrize("size,encoding,n", EXPAND_CASES)
@pytest.mark.parametrize("dtype", (0, 1, 2), ids=DTYPE_IDS)
def test_expand_every_output_set(size, encoding, n, dtype):
    """Every subset of {children, child one-hot, parent one-hot, solved, reward}, with and without counters (a
    subset without one-hot rows runs once, under bf16).  2x2x2 with the exact encoding equals the reference.
    Counters are [solved children, n * A, 0, 0] whenever they are passed; with nothing requested the call
    returns 0."""
    parents = parents_of(size, n)
    want = Want(size, parents, exact=(size == 3 and encoding == 1))
    states = cu(parents)
    for outs in subsets(OUTS):
        if dtype and not outs & ONEHOT_OUTS:
            continue
        for with_counters in (False, True):
            got, counters = run_expand(size, states, outs, dtype, with_counters, encoding)
            check_outputs(want, got, dtype, counters, "%s counters=%s" % (sorted(outs), with_counters))
    assert (states.cpu().numpy() == parents).all()


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("dtype", (0, 1, 2), ids=DTYPE_IDS)
def test_expand_caller_owned_buffers_at_offsets(size, dtype):
    """ops.expand into caller-owned buffers: `solved` at an odd byte, `reward` at 4 mod 16, the one-hot rows as
    16-byte-aligned slices of larger tensors whose other elements must stay untouched.  Both the ADI call (child
    one-hot rows) and the MCTS leaf call (children + parent one-hot rows, no child one-hot rows)."""
    n = EXPAND_N[size][0]
    A, (r, c) = T.N_ACTIONS[size], T.STATE_DIM[size]
    parents = parents_of(size, n, seed=1)
    want = Want(size, parents, exact=False)
    states = cu(parents)
    lead = 3 * 16 // ESIZE[dtype]                               # elements before the slice: 48 bytes
    sentinel = {0: 7.0, 1: 7.0, 2: 7}[dtype]
    for adi in (True, False):
        solved = Guarded(n * A, offset=1)
        reward = Guarded(4 * n * A, torch.float32, offset=4)
        big_c = torch.full((lead + n * A * r * c + lead,), sentinel, dtype=TORCH_DTYPE[dtype], device=dev())
        big_p = torch.full((lead + n * r * c + lead,), sentinel, dtype=TORCH_DTYPE[dtype], device=dev())
        coh = big_c[lead:lead + n * A * r * c].view(n, A, r, c)
        poh = big_p[lead:lead + n * r * c].view(n, r, c)
        res = ops.expand(size, states, dtype=TORCH_DTYPE[dtype], want_children=not adi, want_child_onehot=adi,
                         child_onehot=coh if adi else None, parent_onehot=poh, solved=solved.view, reward=reward.view)
        torch.cuda.synchronize()
        assert solved.intact() and reward.intact()
        assert (solved.view.cpu().numpy() == want.solved.reshape(-1)).all()
        assert (reward.view.cpu().numpy() == want.reward.reshape(-1)).all()
        for big, body, bits in ((big_c, coh, want.child_onehot(dtype)), (big_p, poh, want.parent_onehot(dtype))):
            if body is coh and not adi:
                assert (big == sentinel).all()
                continue
            assert (big[:lead] == sentinel).all() and (big[-lead:] == sentinel).all()
            assert (body.contiguous().view(torch.uint8).cpu().numpy().reshape(-1) == bits).all()
        if not adi:
            assert (res["children"].cpu().numpy() == want.children).all()


# ------------------------------------------------------------------ cube_expand_codes
CODE_OUTS = ("children", "child_codes", "parent_codes", "parent_onehot", "solved", "reward")


@pytest.mark.parametrize("size,encoding,n", [(2, 0, EXPAND_N[2][0]), (2, 0, 11)] +
                         [(3, e, n) for e in (0, 1) for n in EXPAND_N[3]])
def test_expand_codes_every_output_set(size, encoding, n):
    """Every subset of {children, child codes, parent codes, parent one-hot (each dtype), solved, reward}, with and
    without counters.  Codes are the oracle one-hot rows' argmax; the padding bytes are 0."""
    parents = parents_of(size, n, seed=2)
    want = Want(size, parents, exact=(size == 3 and encoding == 1))
    states = cu(parents)
    for outs in subsets(CODE_OUTS):
        for dtype in ((0, 1, 2) if "parent_onehot" in outs else (2,)):
            for with_counters in (False, True):
                got, counters = run_expand_codes(size, states, outs, dtype, with_counters, encoding)
                check_outputs(want, got, dtype, counters, "%s %s counters=%s" % (sorted(outs), DTYPE_IDS[dtype], with_counters))


# ------------------------------------------------------------------ cube_encode
ENCODE_N = (1, 63, 64, 65, 127, 128, 129, 64 * 40 + 37)


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("encoding", ("reference", "exact"))
@pytest.mark.parametrize("dtype", (0, 1, 2), ids=DTYPE_IDS)
def test_encode_into_guarded_buffers(size, encoding, dtype):
    """ops.encode(out=...) at sizes around the 64-row leaf tile and the 128-row encode tile."""
    for n in ENCODE_N:
        parents = parents_of(size, n, seed=3)
        r, c = T.STATE_DIM[size]
        out = Guarded(n * r * c * ESIZE[dtype])
        ops.encode(size, cu(parents), dtype=TORCH_DTYPE[dtype], out=out.view.view(TORCH_DTYPE[dtype]).view(n, r, c),
                   encoding=encoding)
        torch.cuda.synchronize()
        assert out.intact(), n
        assert (host(out) == onehot_bits(size, parents, dtype, size == 3 and encoding == "exact")).all(), n


# ------------------------------------------------------------------ cube_solved
@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("n", (1, 64 * 37 + 29))
def test_solved_every_output_set(size, n):
    """cube_solved with no flags, `solved`, `reward` or both, with and without counters."""
    rows = parents_of(size, n, seed=4)
    rows[::5] = O.solved_states(size, len(rows[::5]))
    want = C.is_solved(size, rows)
    states = cu(rows)
    for has_solved, has_reward in itertools.product((False, True), repeat=2):
        for with_counters in (False, True):
            solved = Guarded(n) if has_solved else None
            reward = Guarded(4 * n) if has_reward else None
            counters = _counters() if with_counters else None
            rc = _lib.load().cube_solved(size, _ptr(states), n, solved and _ptr(solved.view), reward and _ptr(reward.view),
                                         counters and _ptr(counters.view), _stream())
            _lib.check(rc, "cube_solved")
            torch.cuda.synchronize()
            for g in (solved, reward, counters):
                assert g is None or g.intact()
            if solved is not None:
                assert (host(solved) == want.astype(np.uint8)).all()
            if reward is not None:
                assert (host(reward).view(np.float32) == np.where(want, 1.0, -1.0).astype(np.float32)).all()
            if counters is not None:
                assert counters.view.tolist() == [int(want.sum()), n, 0, 0]


# ------------------------------------------------------------------ cube_decode
def decode_ref(size, is_one):
    """The reference's state_to_sim_state per one-hot row: np.where(row == 1)[0][0], column 0 for a row without a 1
    (the library's documented choice; the reference raises there); for 2x2x2 the last cubelet that names a
    position wins (its loop over cubelets), a position nobody names keeps colour 0.  O.decode_2 / O.decode_exact
    apply exactly that to a clean one-hot of these columns."""
    n, r, c = is_one.shape
    first = np.where(is_one.any(axis=2), is_one.argmax(axis=2), 0)
    clean = np.zeros((n, r, c), dtype=np.uint8)
    clean[np.arange(n)[:, None], np.arange(r)[None, :], first] = 1
    return O.decode_2(clean) if size == 2 else O.decode_exact(clean)


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("dtype", (0, 1, 2), ids=DTYPE_IDS)
def test_decode_irregular_rows(size, dtype):
    """ops.decode (2x2x2, 3x3x3 exact) around the 64-row tile, of real one-hot rows and of rows with several 1s,
    no 1, and values that are not 1 (0.5, 2.0, -1.0; in bf16 also the bits 0x3f81, just above 1.0)."""
    r, c = T.STATE_DIM[size]
    for n in (63, 64, 65, 129):
        rng = np.random.RandomState(n + 10 * dtype + size)
        states = parents_of(size, n, seed=5)
        f = (O.encode(2, states) if size == 2 else O.encode_exact(states)).astype(np.float32)
        rows = rng.choice(n, min(n, 40), replace=False)
        for k, i in enumerate(rows):
            cub, col = rng.randint(r), rng.randint(c)
            kind = k % 5
            if kind == 0:
                f[i, cub, col] = 1.0                                    # a second 1 (or the same one)
                f[i, rng.randint(r), rng.randint(c)] = 1.0
            elif kind == 1:
                f[i, cub] = 0.0                                         # no 1
            elif kind == 2:
                f[i, cub] = np.where(f[i, cub] == 1.0, (0.5, 2.0, -1.0)[k % 3], 0.0)
            elif kind == 3:
                f[i, cub, col] = 2.0                                    # argmax would take this one
            else:
                f[i, cub, :] = -1.0
                f[i, cub, c - 1] = 1.0
        bits = f.view(np.uint32) if dtype == 1 else ((f.view(np.uint32) >> 16).astype(np.uint16) if dtype == 0 else
                                                     (f.astype(np.int64) & 0xff).astype(np.uint8))
        if dtype == 0:
            bf = bits.reshape(n, r, c)
            for i in rows[::4]:
                j = int(np.flatnonzero(bf[i, 0] == 0x3f80)[0]) if (bf[i, 0] == 0x3f80).any() else 0
                bf[i, 0, j] = 0x3f81
        is_one = bits.reshape(n, r, c) == ONE[dtype]
        onehot = cu(bits.view(np.uint8).reshape(-1)).view(TORCH_DTYPE[dtype]).view(n, r, c)
        got = ops.decode(size, onehot, encoding="exact" if size == 3 else "reference")
        assert (got.cpu().numpy() == decode_ref(size, is_one)).all(), n
        if size == 2 and dtype == 2:
            clean = O.encode(2, states)                                 # and a real row round-trips
            assert (ops.decode(2, cu(clean).view(n, r, c)).cpu().numpy() == states).all()


# ------------------------------------------------------------------ rows that name a cubelet twice
# (children, child one-hot, parent one-hot, solved) of the calls that reach every 2x2x2 kernel: K3c + generic tail
# (bf16, u8), generic (f32), leaf + generic tail, leaf + encode tail, the generic kernel with every output
TWIN_CALLS = [("children", "child_onehot", "parent_onehot", "solved"), ("child_onehot", "solved"),
              ("children", "parent_onehot", "solved"), ("parent_onehot",), ("child_onehot",)]


@pytest.mark.parametrize("dtype", (0, 1, 2), ids=DTYPE_IDS)
@pytest.mark.parametrize("n", (48, 129, 64 * 40 + 37))
def test_expand_rows_that_name_a_cubelet_twice(dtype, n):
    """The reference's loop (cube_env.py:141-147) gives such a row two 1s in the twice-named cubelet's one-hot row
    and none in the missing cubelet's, wherever the row sits in the batch: every 2x2x2 expansion kernel, cube_encode
    and the codes of cube_expand_codes (argmax: the lowest column set) must say the same."""
    parents = plant_twins(parents_of(2, n, seed=6), seed=n)
    want = Want(2, parents, exact=False)
    states = cu(parents)
    for outs in TWIN_CALLS:
        got, counters = run_expand(2, states, frozenset(outs), dtype, True, 0)
        check_outputs(want, got, dtype, counters, str(outs))
    out = Guarded(n * 147 * ESIZE[dtype])
    ops.encode(2, states, dtype=TORCH_DTYPE[dtype], out=out.view.view(TORCH_DTYPE[dtype]).view(n, 7, 21))
    torch.cuda.synchronize()
    assert out.intact() and (host(out) == want.parent_onehot(dtype)).all()
    got, counters = run_expand_codes(2, states, frozenset(("child_codes", "parent_codes", "parent_onehot")), dtype,
                                     True, 0)
    check_outputs(want, got, dtype, counters, "codes")
    res = ops.expand_codes(2, states)
    assert (res["child_codes"].cpu().numpy().reshape(-1) == want.child_codes()).all()
    assert (res["parent_codes"].cpu().numpy().reshape(-1) == want.parent_codes()).all()


def test_single_cube_encode_of_rows_that_name_a_cubelet_twice():
    """The single-cube front ends (ops.HostCube.encode, the drop-in CubeEnv.sim_state_to_state) on such rows."""
    rows = twin_rows(2, 16, seed=7)
    cube = ops.HostCube(2)
    try:
        for row in rows:
            assert (cube.encode(np.ascontiguousarray(row)) == O.encode(2, row[None])[0]).all()
    finally:
        cube.close()
    env = R.make_env(torch.device("cpu"), 2)
    for row in rows:
        assert (np.asarray(env.sim_state_to_state(row.astype(np.int64))) == O.encode(2, row[None])[0]).all()


# ------------------------------------------------------------------ rows outside the reference's domain
@pytest.mark.parametrize("size", SIZES)
def test_arbitrary_colour_bytes_are_memory_safe(size):
    """Colour bytes >= 6 (the reference's table lookup raises on them): every kernel keeps to its buffers, writes
    one-hot elements 0 or 1, flags 0 or 1, rewards +-1, codes below the row width, and the children stay the plain
    gather."""
    n = EXPAND_N[size][0]
    A, S, D, (r, c), K = T.N_ACTIONS[size], T.N_STICKERS[size], T.ONEHOT_WIDTH[size], T.STATE_DIM[size], ops.key_bytes(size)
    rng = np.random.RandomState(40 + size)
    rows = rng.randint(0, 256, size=(n, S)).astype(np.uint8)
    rows[::2] = rng.randint(0, 8, size=rows[::2].shape)
    states = cu(rows)
    children = rows[:, T.MOVE_DEFS[size]].reshape(-1)
    calls = [(run_expand, outs, dtype, enc) for dtype in (0, 1, 2) for enc in (0, 1)
             for outs in (OUTS, ("child_onehot",), ("children", "parent_onehot", "solved"), ("parent_onehot",))]
    calls += [(run_expand_codes, CODE_OUTS, dtype, enc) for dtype in (0, 1, 2) for enc in (0, 1)]
    for run, outs, dtype, enc in calls:
        got, counters = run(size, states, frozenset(outs), dtype, True, enc)
        what = "%s %s %s" % (run.__name__, sorted(outs), DTYPE_IDS[dtype])
        for name, g in list(got.items()) + [("counters", counters)]:
            assert g.intact(), (what, name)
        if "children" in got:
            assert (host(got["children"]) == children).all(), what
        for name in ONEHOT_OUTS & set(got):
            vals = np.unique(host(got[name]).view(NP_BITS[dtype]))
            assert set(vals.tolist()) <= {0, int(ONE[dtype])}, (what, name, vals[:8])
        if "solved" in got:
            assert set(np.unique(host(got["solved"])).tolist()) <= {0, 1}, what
        if "reward" in got:
            assert set(np.unique(host(got["reward"]).view(np.float32)).tolist()) <= {-1.0, 1.0}, what
        for name in ("child_codes", "parent_codes"):
            if name in got:
                codes = host(got[name]).reshape(-1, K)
                assert (codes[:, :r] < c).all() and (codes[:, r:] == 0).all(), what
        assert counters.view.tolist()[1:] == [n * A, 0, 0], what
    flags = Guarded(n)
    _lib.check(_lib.load().cube_solved(size, _ptr(states), n, _ptr(flags.view), None, None, _stream()), "cube_solved")
    torch.cuda.synchronize()
    assert flags.intact() and (host(flags) == C.is_solved(size, rows).astype(np.uint8)).all()


# ------------------------------------------------------------------ dispatch coverage
def _dispatch_cases():
    """(what the call is, the call, the kernels it must launch)."""
    cases = []
    n2, n3 = EXPAND_N[2][0], EXPAND_N[3][0]
    p2, p3 = cu(parents_of(2, n2, seed=8)), cu(parents_of(3, n3, seed=8))

    def expand(size, states, outs, dtype, enc=0):
        return lambda: run_expand(size, states, frozenset(outs), dtype, False, enc)

    for d, dt in enumerate(("unsigned short", "float", "unsigned char")):
        if d != 1:
            cases.append(("2: ADI %s" % DTYPE_IDS[d], expand(2, p2, ("child_onehot",), d),
                          ["leaf_children_kernel<%d,16>" % d, "expand_kernel<2,%d>" % d]))
        else:
            cases.append(("2: ADI f32", expand(2, p2, ("child_onehot",), d), ["expand_kernel<2,1>"]))
        cases.append(("2: leaf %s" % DTYPE_IDS[d], expand(2, p2, ("children", "parent_onehot"), d),
                      ["leaf_kernel<%d>" % d, "expand_kernel<2,%d>" % d]))
        cases.append(("2: encode %s" % DTYPE_IDS[d], expand(2, p2, ("parent_onehot",), d),
                      ["leaf_kernel<%d>" % d, "encode_kernel<2,%d>" % d]))
        for enc in (0, 1):
            cases.append(("3: expand %s enc %d" % (DTYPE_IDS[d], enc), expand(3, p3, ("child_onehot",), d, enc),
                          ["expand_kernel<3,%d>" % d]))
            cases.append(("3: encode %s enc %d" % (DTYPE_IDS[d], enc), expand(3, p3, ("parent_onehot",), d, enc),
                          ["encode_kernel<3,%d>" % d]))
        oh2 = torch.zeros((n2, 7, 21), dtype=TORCH_DTYPE[d], device=dev())
        oh3 = torch.zeros((n3, 20, 24), dtype=TORCH_DTYPE[d], device=dev())
        cases.append(("2: decode %s" % DTYPE_IDS[d], lambda oh=oh2: ops.decode(2, oh), ["decode2_kernel<%s>" % dt]))
        cases.append(("3: decode %s" % DTYPE_IDS[d], lambda oh=oh3: ops.decode(3, oh, encoding="exact"),
                      ["decode3_exact_kernel<%s>" % dt]))
    cases.append(("2: codes", lambda: ops.expand_codes(2, p2), ["expand_kernel<2,2>"]))
    for size, p in ((2, p2), (3, p3)):
        cases.append(("%d: solved" % size, lambda size=size, p=p: ops.is_solved(size, p), ["walk_tile_kernel<%d," % size]))
    return cases


def missing_kernels():
    """The (case: kernel) lines of _dispatch_cases whose kernel a trace of the case does not show, or None when
    torch.profiler recorded no CUDA activity at all (CUPTI unavailable)."""
    from torch.profiler import ProfilerActivity, profile
    cases = _dispatch_cases()
    for _, call, _ in cases:                                # first launches (attributes, modules) outside the trace
        call()
    torch.cuda.synchronize()
    seen_any = False
    missing = []
    for what, call, expect in cases:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            call()
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        seen_any = seen_any or bool(names)
        keys = {_kernel_key(s) for s in names} - {None}
        missing += ["%s: %s (launched: %s)" % (what, k, sorted(keys)) for k in expect
                    if not any(x == k or (k.endswith(",") and x.startswith(k)) for x in keys)]
    return missing if seen_any else None


def test_dispatch_reaches_every_expansion_kernel():
    """Each case launches the kernels the dispatch table above names (recorded with torch.profiler), so a dispatch
    change cannot move this file's coverage away unnoticed.  `walk_tile_kernel<S,` is matched as a prefix.  The
    trace runs in an interpreter of its own: in one process with test_optional_outputs_gpu.py's dispatch test, the
    profiler sessions of the one that ran first made the other's sessions record no kernels."""
    if "CUBE_K3C_TILE" in os.environ:
        pytest.skip("CUBE_K3C_TILE changes the dispatch")
    here = os.path.dirname(os.path.abspath(__file__))
    script = ("import sys; sys.path[:0] = [%r, %r]\n"
              "import test_expand_outputs_gpu as t\n"
              "m = t.missing_kernels()\n"
              "print('NO CUDA ACTIVITY' if m is None else '\\n'.join(m) or 'ALL LAUNCHED')\n") % (os.path.dirname(here), here)
    out = subprocess.run([sys.executable, "-c", script], capture_output=True, text=True, timeout=600,
                         cwd=os.path.dirname(here))
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    if out.stdout.strip().endswith("NO CUDA ACTIVITY"):
        pytest.skip("torch.profiler recorded no CUDA activity (CUPTI unavailable): kernel dispatch not checked")
    assert out.stdout.strip().endswith("ALL LAUNCHED"), out.stdout[-4000:]
