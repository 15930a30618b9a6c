"""The optional outputs of the scramble, scramble-step and walk kernels against the oracle.

The batch launchers pick a kernel instantiation from the depth, the buffers' alignment and WHICH optional outputs
the caller passed: K1p (scramble_pairs_kernel) compiles the null checks out when `solved` and `reward` are both
present (MODE 1, MODE 2 with the trailing action of cube_scramble_step) and decides at run time otherwise
(MODE 0); the sliced, tile, deep, K2p (walk_private_kernel) and walk tile kernels test every pointer at run time.
Every output set (no flags, `solved` only, `reward` only, both; with and without counters) runs here on every
variant, with every present output between guard bytes, and is compared bit for bit with the C oracle.  The
production callers that leave flags out (rollout's greedy solve and validation, the host pipeline) run at their
own shapes, and one test checks with torch.profiler that the cases reach every kernel instantiation."""
import ctypes
import functools
import os
import re

import numpy as np
import pytest
import torch

from rubiks_cube_solver_b200 import _lib, ops, rollout

from oracle import cube_c as C
from oracle import tables as T

pytestmark = pytest.mark.gpu
SIZES = (2, 3)
NOOP = 12                                                  # CUBE_NOOP: indices A..12 leave the cube unchanged
FILL = 0xA5
FLAG_SETS = {"none": (False, False), "solved": (True, False), "reward": (False, True), "both": (True, True)}


def dev():
    return torch.device("cuda", 0)


def cu(a, dtype=np.uint8):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=dtype)).to(dev())


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream(dev()).cuda_stream)


class Guarded(object):
    """`n_bytes` of payload with 4096 canary bytes on both sides, `offset` bytes past a 16-byte boundary.
    On the device unless `host` (then page-locked)."""

    def __init__(self, n_bytes, dtype=torch.uint8, offset=0, host=False, guard=4096):
        size = guard + n_bytes + 31 + guard
        if host:
            self.raw = torch.full((size,), FILL, dtype=torch.uint8).pin_memory()
        else:
            self.raw = torch.full((size,), FILL, dtype=torch.uint8, device=dev())
        self.lo = guard + (-(self.raw.data_ptr() + guard)) % 16 + offset
        self.n_bytes = n_bytes
        self.view = self.raw[self.lo:self.lo + n_bytes].view(dtype)

    def intact(self):
        return bool((self.raw[:self.lo] == FILL).all()) and bool((self.raw[self.lo + self.n_bytes:] == FILL).all())


def _counters():
    g = Guarded(32, torch.int64)
    g.view.zero_()
    return g


def oracle(size, moves, init=None):
    """(states, solved, reward) of the C oracle for `moves` from solved (or from `init`); a move index in A..12 is
    the no-op, as in the kernels (include/cube_b200.h).  Rows are grouped by their number of real moves."""
    moves = np.ascontiguousarray(moves, dtype=np.uint8)
    assert moves.size == 0 or moves.max() <= NOOP
    keep = moves < T.N_ACTIONS[size]
    if keep.all():
        return C.scramble(size, moves, init=init)[:3]
    n = moves.shape[0]
    states = np.empty((n, T.N_STICKERS[size]), dtype=np.uint8)
    solved = np.empty(n, dtype=bool)
    reward = np.empty(n, dtype=np.float32)
    lens = keep.sum(axis=1)
    for k in np.unique(lens):
        rows = np.flatnonzero(lens == k)
        m = moves[rows][keep[rows]].reshape(len(rows), int(k))
        states[rows], solved[rows], reward[rows], _ = C.scramble(size, m, init=None if init is None else init[rows])
    return states, solved, reward


def batch_rows(size):
    """Whole K1p tiles -- 64 rows, 128 for a 2x2x2 with four instances per lane -- at least three per CTA of a
    full-width launch, and a ragged tail for the tile / deep kernels."""
    return (64 if size == 3 else 128) * 148 * 3 + 37


def plant_identities(moves, rows):
    """Make `rows` of `moves` come back to solved: half the row, its inverse, and a no-op when the depth is odd
    (a quarter-turn identity has even length)."""
    depth = moves.shape[1]
    h = depth // 2
    moves[rows, h:2 * h] = moves[rows, :h][:, ::-1] ^ 1
    if depth % 2:
        moves[rows, -1] = NOOP


@functools.lru_cache(maxsize=None)
def scramble_case(size, depth, n, seed=0):
    """Seeded moves with rows that end solved (the first 64, 300 random ones, the last three) and the oracle."""
    rng = np.random.RandomState(1000 * size + depth + seed)
    moves = rng.randint(T.N_ACTIONS[size], size=(n, depth)).astype(np.uint8)
    back = np.concatenate((np.arange(64), rng.choice(n, 300, replace=False), np.arange(n - 3, n)))
    plant_identities(moves, back)
    want = oracle(size, moves)
    assert want[1][back].all()
    return moves, want


def run_scramble(size, moves, flags, with_counters, solved_offset=0, reward_offset=0):
    """ops.scramble with the outputs `flags` names, each between guard bytes; returns the buffers."""
    n, S = moves.shape[0], T.N_STICKERS[size]
    has_solved, has_reward = FLAG_SETS[flags]
    out = Guarded(n * S)
    solved = Guarded(n, offset=solved_offset) if has_solved else None
    reward = Guarded(4 * n, torch.float32, offset=reward_offset) if has_reward else None
    counters = _counters() if with_counters else None
    states, so, rw = ops.scramble(size, cu(moves), out=out.view.view(n, S), solved=solved and solved.view,
                                  reward=reward and reward.view, counters=counters and counters.view, want_flags=False)
    assert (so is None) == (solved is None) and (rw is None) == (reward is None)
    torch.cuda.synchronize()
    return out, solved, reward, counters


def check(want, out, solved, reward, counters):
    """Every present output equals the oracle bit for bit and nothing around it was written."""
    ws_states, ws, wr = want
    n = len(ws)
    for g in (out, solved, reward, counters):
        assert g is None or g.intact()
    assert (out.view.view(n, -1).cpu().numpy() == ws_states).all()
    if solved is not None:
        assert (solved.view.cpu().numpy() == ws.astype(np.uint8)).all()
    if reward is not None:
        assert (reward.view.cpu().numpy() == wr).all()
    if counters is not None:
        assert counters.view.tolist() == [int(ws.sum()), n, 0, 0]


# ------------------------------------------------------------------ cube_scramble (ops.scramble)
# 1, 31: K1p's generic kernel; 20, 30: its straight-line kernels; 24: swizzled for the 3x3x3, generic for the
# 2x2x2; 32: swizzled for both; 160 / 161: the deepest tail the tile kernel stages and the first that goes to the
# deep kernel; 321 / 400: the sliced kernel, with its last whole tile and the tail in the deep kernel
SCRAMBLE_DEPTHS = (1, 20, 24, 30, 31, 32, 160, 161, 321, 400)


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("depth", SCRAMBLE_DEPTHS)
@pytest.mark.parametrize("flags", list(FLAG_SETS))
@pytest.mark.parametrize("with_counters", (False, True), ids=("nocnt", "cnt"))
def test_scramble_every_output_set(size, depth, flags, with_counters):
    """Each output set on each scramble variant; with the flags off the counters still count."""
    moves, want = scramble_case(size, depth, batch_rows(size))
    check(want, *run_scramble(size, moves, flags, with_counters))


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("depth", (20, 30, 32))
@pytest.mark.parametrize("flags", ("none", "solved", "reward"))
def test_scramble_output_sets_many_tiles_per_warp(size, depth, flags):
    """MODE 0 of K1p on two persistent CTAs: every warp walks many tiles (both move buffers, the barriers' phases,
    the dynamic tail), each with its run-time null checks."""
    moves, want = scramble_case(size, depth, 64 * 900 + 17, seed=1)
    ops.set_reserved_sms(ops.sm_count() - 2)
    try:
        got = run_scramble(size, moves, flags, True)
    finally:
        ops.set_reserved_sms(0)
    check(want, *got)


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("depth", (30, 400))
@pytest.mark.parametrize("flags,solved_offset,reward_offset", [("solved", 1, 0), ("reward", 0, 4)],
                         ids=("solved_odd", "reward_4"))
def test_scramble_partial_flags_unaligned(size, depth, flags, solved_offset, reward_offset):
    """One flag array alone, not aligned for K1p's paired stores (`solved` at an odd byte, `reward` 4- but not
    8-byte aligned): the whole batch goes to the byte-wise tile kernel (depth 30) or the deep kernel (400)."""
    moves, want = scramble_case(size, depth, batch_rows(size))
    got = run_scramble(size, moves, flags, True, solved_offset=solved_offset, reward_offset=reward_offset)
    check(want, *got)


# ------------------------------------------------------------------ cube_scramble_step (C ABI)
def _step_case(size, depth, n):
    """Moves and trailing actions with rows whose scramble + action is the identity: for an even depth the
    scramble is an identity and the action the no-op, for an odd one the action undoes the last move."""
    rng = np.random.RandomState(7 * depth + size)
    A = T.N_ACTIONS[size]
    moves = rng.randint(A, size=(n, depth)).astype(np.uint8)
    act = rng.randint(A, size=n).astype(np.uint8)
    back = np.concatenate((np.arange(64), rng.choice(n, 300, replace=False), np.arange(n - 3, n)))
    seq = np.concatenate((moves, act[:, None]), axis=1)
    h = (depth + 1) // 2
    seq[back, h:2 * h] = seq[back, :h][:, ::-1] ^ 1
    if (depth + 1) % 2:
        seq[back, -1] = NOOP
    moves, act = np.ascontiguousarray(seq[:, :depth]), np.ascontiguousarray(seq[:, depth])
    return moves, act, oracle(size, seq), back


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("depth", (0, 1, 20, 30, 32, 321))
@pytest.mark.parametrize("flags", list(FLAG_SETS))
def test_scramble_step_abi_output_sets(size, depth, flags):
    """cube_scramble_step with each output set (ops.scramble_step always passes both flags): the only way to
    reach K1p's MODE 0 with a trailing action for the 3x3x3.  Oracle: the scramble, then the action."""
    n, S = batch_rows(size), T.N_STICKERS[size]
    moves, act, want, back = _step_case(size, depth, n)
    assert want[1][back].all()
    has_solved, has_reward = FLAG_SETS[flags]
    out = Guarded(n * S)
    solved = Guarded(n) if has_solved else None
    reward = Guarded(4 * n, torch.float32) if has_reward else None
    counters = _counters()
    m, a = cu(moves), cu(act)
    rc = _lib.load().cube_scramble_step(size, _ptr(m) if depth else None, _ptr(a), n, depth, _ptr(out.view),
                                        solved and _ptr(solved.view), reward and _ptr(reward.view),
                                        _ptr(counters.view), _stream())
    _lib.check(rc, "cube_scramble_step")
    torch.cuda.synchronize()
    check(want, out, solved, reward, counters)


# ------------------------------------------------------------------ cube_walk / cube_step (C ABI)
@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("depth", (1, 5, 64, 65))
@pytest.mark.parametrize("flags", list(FLAG_SETS))
def test_walk_and_step_abi_output_sets(size, depth, flags):
    """cube_walk out of place and in place (cube_step in place at depth 1) with each output set (ops.walk and
    ops.step always pass both flags): K2p at depth <= 64, the walk tile kernel beyond and for the tail."""
    rng = np.random.RandomState(31 * depth + size)
    A, S = T.N_ACTIONS[size], T.N_STICKERS[size]
    n = 64 * 148 * 2 + 29
    moves = rng.randint(A, size=(n, depth)).astype(np.uint8)
    start = oracle(size, rng.randint(A, size=(n, 9)))[0]
    back = np.concatenate((np.arange(64), rng.choice(n, 300, replace=False), np.arange(n - 3, n)))
    start[back] = oracle(size, moves[back, ::-1] ^ 1)[0]               # the walk undoes these starts
    want = oracle(size, moves, init=start)
    assert want[1][back].all()
    has_solved, has_reward = FLAG_SETS[flags]
    lib = _lib.load()
    m = cu(moves)
    for in_place in (False, True):
        states_in = Guarded(n * S)
        states_in.view.copy_(cu(start).view(-1))
        out = states_in if in_place else Guarded(n * S)
        solved = Guarded(n) if has_solved else None
        reward = Guarded(4 * n, torch.float32) if has_reward else None
        counters = _counters()
        flag_ptrs = (solved and _ptr(solved.view), reward and _ptr(reward.view), _ptr(counters.view), _stream())
        if in_place and depth == 1:
            rc = lib.cube_step(size, _ptr(out.view), _ptr(m), n, *flag_ptrs)
        else:
            rc = lib.cube_walk(size, _ptr(states_in.view), _ptr(m), n, depth, _ptr(out.view), *flag_ptrs)
        _lib.check(rc, "cube_step" if in_place and depth == 1 else "cube_walk")
        torch.cuda.synchronize()
        check(want, out, solved, reward, counters)
        assert in_place or (states_in.view.cpu().numpy() == start.reshape(-1)).all()


# ------------------------------------------------------------------ production shapes
@pytest.mark.parametrize("size,depth", [(3, 30), (2, 20)])
def test_noop_padded_reference_scrambles_without_flags(size, depth):
    """rollout.validation's scrambles: reset(seed, d) for d = 1..depth, padded with the no-op index to one depth,
    scrambled with want_flags=False as greedy_solve does -- K1p's MODE 0 straight-line kernel."""
    seeds = list(range(0, 10000, 10))
    moves = rollout.reference_scrambles_device(size, seeds, range(1, depth + 1))
    host = moves.cpu().numpy()
    for d in (1, depth // 2, depth):
        for j in (0, 1, len(seeds) - 1):
            row = host[(d - 1) * len(seeds) + j]
            assert (row[:d] == np.random.RandomState(seeds[j]).randint(T.N_ACTIONS[size], size=d)).all()
            assert (row[d:] == NOOP).all()
    states, solved, reward = ops.scramble(size, moves, want_flags=False)
    assert solved is None and reward is None
    assert (states.cpu().numpy() == oracle(size, host)[0]).all()


@functools.lru_cache(maxsize=None)
def _seeded_moves(size, seeds, depth):
    return np.stack([np.random.RandomState(s).randint(T.N_ACTIONS[size], size=depth) for s in seeds]).astype(np.uint8)


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("n_stages", (1, 2, 3, 4))
@pytest.mark.parametrize("want_solved,want_reward", [(False, False), (True, False), (False, True), (True, True)],
                         ids=("none", "solved", "reward", "both"))
def test_host_pipeline_flag_combinations(size, n_stages, want_solved, want_reward):
    """HostScramblePipeline.run and .reset with each (want_solved, want_reward): a flag left out reaches the kernel
    as a null pointer.  Chunks of 1 000 instances (rounded up to 1 024), a ragged last chunk, every stage reused;
    outputs in caller-owned host buffers between guard bytes.  .reset at depth 4, where seeds come back solved."""
    n, S, A = 1024 * 5 + 77, T.N_STICKERS[size], T.N_ACTIONS[size]
    cases = []
    moves, want = scramble_case(size, 30 if size == 3 else 20, n, seed=2)
    cases.append(("run", torch.from_numpy(moves).pin_memory(), moves.shape[1], want))
    seeds = tuple(range(3, 3 + 7 * n, 7))
    want_reset = oracle(size, _seeded_moves(size, seeds, 4))
    assert want_reset[1].any()
    cases.append(("reset", torch.tensor(seeds, dtype=torch.int32), 4, want_reset))
    for how, inputs, depth, want in cases:
        out = Guarded(n * S, host=True)
        solved = Guarded(n, host=True) if want_solved else None
        reward = Guarded(4 * n, torch.float32, host=True) if want_reward else None
        pipe = ops.HostScramblePipeline(size, depth, chunk_instances=1000, n_stages=n_stages)
        try:
            states, so, rw, count = getattr(pipe, how)(inputs, states_out=out.view.view(n, S),
                                                       solved=solved and solved.view, reward=reward and reward.view,
                                                       want_solved=want_solved, want_reward=want_reward)
        finally:
            pipe.close()
        assert (so is None) != want_solved and (rw is None) != want_reward
        check(want, out, solved, reward, None)
        assert count == int(want[1].sum()), how


# ------------------------------------------------------------------ dispatch coverage
_DISPATCH_SWITCHES = ("CUBE_SCRAMBLE_CLASSIC", "CUBE_PAIR_FOUR", "CUBE_PAIR_SWIZZLE", "CUBE_PAIR_SLICED",
                      "CUBE_WALK_CLASSIC")


def _kernel_key(name):
    """'scramble_pairs_kernel<3,-1,2,0>' from a demangled kernel name, whichever way the demangler prints
    template arguments ('(int)-1', 'true'); None for other kernels."""
    m = re.search(r"(\w+_kernel)<([^<>]*)>", name)
    if not m:
        return None
    args = [re.sub(r"^\((?:int|bool)\)", "", a.strip()) for a in m.group(2).split(",")]
    args = [{"true": "1", "false": "0"}.get(a, a) for a in args]
    return "%s<%s>" % (m.group(1), ",".join(args))


def _dispatch_cases():
    """(what the call is, the call, the kernels it must launch) for every row of the dispatch table."""
    n = 64 * 20 + 37                                       # 20 tiles of 64 (10 of 128) + a 37-row tail
    cases = []

    def scramble(size, depth, flags, step=False, solved_offset=0):
        moves = cu(np.random.RandomState(depth).randint(T.N_ACTIONS[size], size=(n, depth)))
        has_solved, has_reward = FLAG_SETS[flags]
        solved = Guarded(n, offset=solved_offset).view if has_solved else None
        reward = torch.empty(n, dtype=torch.float32, device=dev()) if has_reward else None
        out = torch.empty((n, T.N_STICKERS[size]), dtype=torch.uint8, device=dev())
        if step:
            act = torch.zeros(n, dtype=torch.uint8, device=dev())
            return lambda: _lib.check(_lib.load().cube_scramble_step(size, _ptr(moves), _ptr(act), n, depth, _ptr(out),
                                                                    _ptr(solved), _ptr(reward), None, _stream()), "step")
        return lambda: ops.scramble(size, moves, out=out, solved=solved, reward=reward, want_flags=False)

    def walk(size, depth):
        moves = cu(np.random.RandomState(depth).randint(T.N_ACTIONS[size], size=(n, depth)))
        states = ops.solved_states(size, n, dev())
        return lambda: ops.walk(size, states, moves)

    # 3x3x3, two instances per lane: generic (31), straight-line (30, 20), swizzled (32) x MODE 1 / 0 / 2
    for depth, d in ((31, 0), (30, 30), (20, 20), (32, -1)):
        for flags, step, mode in (("both", False, 1), ("none", False, 0), ("reward", False, 0), ("both", True, 2),
                                  ("none", True, 0)):
            cases.append(("3x3x3 depth %d %s%s" % (depth, flags, " +action" if step else ""), scramble(3, depth, flags, step),
                          ["scramble_pairs_kernel<3,%d,2,%d>" % (d, mode)]))
    # 2x2x2: four per lane at shallow depths (swizzled at 16), two per lane deeper; its trailing-action calls are MODE 0
    for depth, d, ns in ((31, 0, 4), (30, 30, 4), (20, 20, 4), (16, -1, 4), (161, 0, 2), (32, -1, 2)):
        for flags, step, mode in (("both", False, 1), ("solved", False, 0), ("both", True, 0)):
            cases.append(("2x2x2 depth %d %s%s" % (depth, flags, " +action" if step else ""), scramble(2, depth, flags, step),
                          ["scramble_pairs_kernel<2,%d,%d,%d>" % (d, ns, mode)]))
    for size in SIZES:
        cases.append(("%d: depth 400" % size, scramble(size, 400, "both"),
                      ["scramble_sliced_kernel<%d>" % size, "scramble_deep_kernel<%d>" % size]))
        cases.append(("%d: depth 30, solved at an odd address" % size, scramble(size, 30, "solved", solved_offset=1),
                      ["scramble_tile_kernel<%d,1>" % size, "scramble_tile_kernel<%d,0>" % size]))
        cases.append(("%d: walk depth 1" % size, walk(size, 1),
                      ["walk_private_kernel<%d>" % size, "walk_tile_kernel<%d,0>" % size]))
        cases.append(("%d: walk depth 65" % size, walk(size, 65), ["walk_tile_kernel<%d,1>" % size]))
    return cases


def test_dispatch_reaches_every_kernel_variant():
    """Each row of the dispatch table -- scramble_pairs_kernel<SIZE, DEPTH, NS, MODE> for every MODE and variant the
    default dispatch reaches (the 2x2x2 two-per-lane straight-line kernels only run under CUBE_PAIR_FOUR=0), the
    sliced, tile (full and tail) and deep scramble kernels, K2p and the walk tile kernel -- is launched by a
    representative call, recorded with torch.profiler.  Keeps a dispatch change from moving this file's coverage
    away unnoticed."""
    from torch.profiler import ProfilerActivity, profile
    set_switches = [s for s in _DISPATCH_SWITCHES if s in os.environ]
    if set_switches:
        pytest.skip("A/B switches %s change the dispatch" % ", ".join(set_switches))
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
        keys = {_kernel_key(s) for s in names}
        missing += ["%s: %s (launched: %s)" % (what, k, sorted(x for x in keys if x)) for k in expect if k not in keys]
    if not seen_any:
        pytest.skip("torch.profiler recorded no CUDA activity (CUPTI unavailable): kernel dispatch not checked")
    assert not missing, "\n".join(missing)
