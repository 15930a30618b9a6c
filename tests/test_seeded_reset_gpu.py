"""Seeded resets on every front end against NumPy's legacy generator and the oracle: reset(seed, k) is
np.random.seed(seed); np.random.randint(A, size=k) and k moves from solved (cube_env.py:61-69).

K0 (cube_moves_from_seeds) draws the first 227 raw outputs of a seed's generator without its state and takes
an exact slow path for a row those leave short; the seeds below are the only ones < 2**32 where that happens at
depth <= 128.  Deeper scrambles go through the host fallbacks (depth > 128) and the single-cube kernel's
64-move chunks (CubeEnv, HostCube)."""
import ctypes

import numpy as np
import pytest
import torch

import rubiks_cube_solver_b200 as R
from rubiks_cube_solver_b200 import _lib, ops, rollout

from oracle import cube_c as C
from oracle import cube_np as O
from oracle import tables as T

pytestmark = pytest.mark.gpu
SIZES = (2, 3)
FAST_DRAWS = 227
STARVED = [2103926524, 3830291768, 3969546545]        # randint(12): 125, 127 accepted of 227; randint(6): 126
GUARD = 0xA5


def dev():
    return torch.device("cuda", 0)


def _accepted_in_fast_draws(cube_size, seed):
    raw = np.random.RandomState(seed).randint(0, 2 ** 32, size=FAST_DRAWS, dtype=np.uint32)
    return int(((raw & (15 if cube_size == 3 else 7)) <= (11 if cube_size == 3 else 5)).sum())


def _packed(seeds):
    return torch.from_numpy(np.asarray(seeds, dtype=np.int64).astype(np.uint32).view(np.int32).copy())


def _batches(size):
    """Seed batches that put slow-path rows next to fast ones: three lanes of one warp, the ragged last CTA of
    128 rows, and each starved seed alone."""
    rng = np.random.RandomState(40 + size)
    warp = rng.randint(0, 2 ** 32, size=96, dtype=np.uint64).astype(np.int64)
    warp[[37, 38, 53]] = STARVED
    ragged = rng.randint(0, 2 ** 32, size=3 * 128 + 45, dtype=np.uint64).astype(np.int64)
    ragged[:4] = [0, 2 ** 31 - 1, 2 ** 31, 2 ** 32 - 1]
    ragged[[384, 400, 428]] = STARVED
    return [warp, ragged] + [np.array([s], dtype=np.int64) for s in STARVED]


@pytest.mark.parametrize("size", SIZES)
def test_moves_from_seeds_slow_path_rows_at_every_depth(size):
    """Every depth 1..128, output between guard bytes: slow lanes beside fast ones in a warp, in the ragged last
    CTA and alone are NumPy's rows, nothing outside the rows is written, counters[3] counts the slow rows."""
    a = T.N_ACTIONS[size]
    lib = _lib.load()
    batches = _batches(size)
    assert min(_accepted_in_fast_draws(size, s) for s in STARVED) < 128          # the slow path runs for this size
    for seeds in batches:
        want = np.stack([np.random.RandomState(int(s)).randint(a, size=128) for s in seeds])
        accepted = np.array([_accepted_in_fast_draws(size, int(s)) for s in seeds])
        d_seeds = _packed(seeds).to(dev())
        n = len(seeds)
        for depth in range(1, 129):
            nbytes = n * depth
            raw = torch.full((4096 + nbytes + 15 + 4096,), GUARD, dtype=torch.uint8, device=dev())
            lo = 4096 + (-(raw.data_ptr() + 4096)) % 16
            counters = ops.new_counters(dev())
            rc = lib.cube_moves_from_seeds(size, ctypes.c_void_p(d_seeds.data_ptr()), n, depth,
                                           ctypes.c_void_p(raw.data_ptr() + lo), ctypes.c_void_p(counters.data_ptr()), None)
            assert rc == 0
            torch.cuda.synchronize()
            host = raw.cpu().numpy()
            assert (host[lo:lo + nbytes].reshape(n, depth) == want[:, :depth]).all(), (n, depth)
            assert (host[:lo] == GUARD).all() and (host[lo + nbytes:] == GUARD).all(), (n, depth)
            assert counters.tolist() == [0, 0, 0, int((accepted < depth).sum())], (n, depth)
    # the torch wrapper: no error for slow rows, the same counter
    counters = ops.new_counters(dev())
    got = ops.moves_from_seeds(size, batches[1], 128, counters=counters)
    want = np.stack([np.random.RandomState(int(s)).randint(a, size=128) for s in batches[1]])
    assert (got.cpu().numpy() == want).all()
    assert int(counters[3]) == sum(_accepted_in_fast_draws(size, int(s)) < 128 for s in batches[1])


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("depth", (127, 128, 129))
def test_batched_env_reset_from_seeds_at_and_past_depth_128(size, depth):
    """BatchedCubeEnv.reset(seeds, k): drawn on the device up to k = 128, on the host beyond."""
    seeds = STARVED + list(range(0, 4000, 10)) + [2 ** 32 - 1]
    env = R.BatchedCubeEnv(len(seeds), cube_size=size, obs_dtype=torch.float32)
    obs, reward, done = env.reset(seeds=seeds, scramble_count=depth)
    want = O.scramble(size, np.stack([O.reference_moves(size, s, depth) for s in seeds]))
    want_solved = O.is_solved(size, want)
    assert (env.sim_cube.cpu().numpy() == want).all()
    assert (obs.cpu().numpy() == O.encode(size, want)).all()
    assert (done.cpu().numpy().astype(bool) == want_solved).all()
    assert (reward.cpu().numpy() == O.rewards(want_solved)).all()


# 2x2x2 seeds whose reset(seed, 128) ends on the solved cube (found by a search over the first 2^25 seeds)
SOLVED_AT_128 = [3064279, 3736840]


@pytest.mark.parametrize("size", SIZES)
def test_host_reset_pipeline_with_slow_path_seeds_in_different_chunks(size):
    """cube_pipeline_reset_host at depth 128: the slow-path seeds in chunks 0, 1, 3 and the ragged last one."""
    rng = np.random.RandomState(50 + size)
    n = 5 * 1024 + 77
    seeds = rng.randint(0, 2 ** 32, size=n, dtype=np.uint64).astype(np.int64)
    seeds[[3, 1024 + 500, 3 * 1024 + 1, n - 1]] = STARVED + [STARVED[0]]
    if size == 2:
        seeds[[10, 4000]] = SOLVED_AT_128
    moves = np.stack([O.reference_moves(size, int(s), 128) for s in seeds]).astype(np.uint8)
    want, want_solved, want_reward, _ = C.scramble(size, moves)
    pipe = ops.HostScramblePipeline(size, 128, chunk_instances=1024, n_stages=3)
    try:
        states, solved, reward, count = pipe.reset(_packed(seeds))
    finally:
        pipe.close()
    assert (states.numpy() == want).all()
    assert (solved.numpy().astype(bool) == want_solved).all() and (reward.numpy() == want_reward).all()
    assert count == int(want_solved.sum()) == (2 if size == 2 else 0)


@pytest.mark.parametrize("size", SIZES)
def test_reference_scrambles_device_around_depth_128(size):
    """rollout.reference_scrambles_device against the host draw: one K0 row per seed cut to every depth up to
    128, the host draw beyond -- on the device either way."""
    seeds = STARVED + [0, 10, 20, 2 ** 32 - 1]
    for depths in ([1, 30, 125, 126, 127, 128], [5, 127, 128, 129]):
        got = rollout.reference_scrambles_device(size, seeds, depths)
        assert got.is_cuda and got.dtype == torch.uint8
        assert (got.cpu().numpy() == rollout.reference_scrambles(size, seeds, depths)).all()


@pytest.mark.parametrize("size", SIZES)
def test_drop_in_reset_long_and_slow_path_scrambles(size):
    """CubeEnv.reset(seed, k) for k around the single-cube kernel's 64-move chunks, test.py's 1 000, the 1 024 of
    its session and the device-tensor fallback beyond; the global NumPy generator is left as it was."""
    env = R.make_env(torch.device("cpu"), size)
    assert env._host().max_depth == 1024                                       # 1025 takes the fallback
    np.random.seed(7)
    before = np.random.get_state()
    cases = [(s, k) for k in (63, 64, 65, 128, 129, 1000, 1024, 1025) for s in (0, 10, 2 ** 32 - 1)]
    for seed, k in cases + [(s, 128) for s in STARVED]:
        obs = env.reset(seed, k)
        want = O.scramble(size, O.reference_moves(size, seed, k)[None])
        assert env.sim_cube.dtype == np.int64 and (env.sim_cube == want[0]).all(), (seed, k)
        assert obs is env.cube and obs.dtype == (np.float64 if size == 2 else np.int64)
        assert (obs == O.encode(size, want)[0]).all(), (seed, k)
    after = np.random.get_state()
    assert before[0] == after[0] and (before[1] == after[1]).all() and before[2:] == after[2:]


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("depth", (1, 64, 65, 4001, 4096))
def test_host_cube_deep_scrambles_with_noop_indices(size, depth):
    """HostCube(max_depth=4096).scramble: the single-cube kernel's 64-move chunks up to 4 096 moves, with every
    no-op index A..12 among them, against the oracle's scramble of the moves without the no-ops."""
    a = T.N_ACTIONS[size]
    rng = np.random.RandomState(depth * 3 + size)
    moves = rng.randint(a, size=depth).astype(np.uint8)
    noop = rng.rand(depth) < 0.1
    moves[noop] = rng.randint(a, 13, size=int(noop.sum()))
    if depth >= 13 - a:
        moves[rng.choice(depth, 13 - a, replace=False)] = np.arange(a, 13)
    # one more scramble of the same length that comes back to solved: half a walk, its inverse, no-ops between
    half = rng.randint(a, size=(depth - depth // 10) // 2).astype(np.uint8)
    walk = np.concatenate([half, half[::-1] ^ 1])
    back = np.insert(walk, np.sort(rng.randint(0, len(walk) + 1, size=depth - len(walk))),
                     rng.randint(a, 13, size=depth - len(walk))).astype(np.uint8)
    hc = ops.HostCube(size, max_depth=4096)
    try:
        for seq in (moves, back):
            stickers, onehot, solved = hc.scramble(seq)
            want = O.scramble(size, seq[seq < a][None])
            assert (stickers == want[0]).all() and (onehot == O.encode(size, want)[0]).all()
            assert solved == bool(O.is_solved(size, want)[0])
        assert hc.scramble(back)[2]
    finally:
        hc.close()
