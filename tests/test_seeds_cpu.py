"""K0's per-seed draw without a GPU: csrc/cube_seeds.cuh compiled with g++ (tests/host_emul/seeds_emul.cpp) against
NumPy's legacy generator, `np.random.RandomState(seed).randint(A, size=depth)` -- what reset(seed, depth) draws
(cube_env.py:62-65) -- at every depth 1..128, for the seeds whose first 227 raw outputs hold too few accepted
values (the slow path) and for a few thousand others."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))

FAST_DRAWS = 227                       # raw outputs K0 draws without materialising the generator state
# (cube_size, seed, values randint(A) accepts among the first 227 raw outputs): the only seeds < 2**32 short of 128
STARVED = [(3, 2103926524, 125), (3, 3830291768, 127), (2, 3969546545, 126)]
EDGE_SEEDS = [0, 1, 2 ** 31 - 1, 2 ** 31, 2 ** 32 - 1]
DEPTHS = range(1, 129)


def _accepted_in_fast_draws(cube_size, seed):
    """How many of the first 227 raw 32-bit outputs randint(A)'s masked rejection accepts (NumPy alone)."""
    raw = np.random.RandomState(seed).randint(0, 2 ** 32, size=FAST_DRAWS, dtype=np.uint32)
    max_value = 11 if cube_size == 3 else 5
    mask = 15 if cube_size == 3 else 7
    return int(((raw & mask) <= max_value).sum())


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    lib_path = str(tmp_path_factory.mktemp("seeds_emul") / "libseeds_emul.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-w", "-o", lib_path,
                           os.path.join(HERE, "host_emul", "seeds_emul.cpp")])
    lib = ctypes.CDLL(lib_path)
    lib.emul_moves_from_seeds.argtypes = [ctypes.c_int, ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int, ctypes.c_void_p]
    lib.emul_moves_from_seeds.restype = ctypes.c_longlong
    return lib


def _draw(emul, cube_size, seeds, depth):
    seeds = np.ascontiguousarray(seeds, dtype=np.uint32)
    out = np.full((len(seeds), depth), 0xee, dtype=np.uint8)
    slow = emul.emul_moves_from_seeds(cube_size, seeds.ctypes.data, len(seeds), depth, out.ctypes.data)
    return out, slow


def test_starved_seeds_need_more_than_227_raw_draws():
    for size, seed, accepted in STARVED:
        assert _accepted_in_fast_draws(size, seed) == accepted < 128


@pytest.mark.parametrize("size", (2, 3))
def test_emulated_draws_of_starved_seeds_equal_numpy(emul, size):
    a = 12 if size == 3 else 6
    seeds = [s for _, s, _ in STARVED]
    accepted = [_accepted_in_fast_draws(size, s) for s in seeds]
    assert min(accepted) < 128                                # the slow path runs for this size
    for depth in DEPTHS:
        got, slow = _draw(emul, size, seeds, depth)
        want = np.stack([np.random.RandomState(s).randint(a, size=depth) for s in seeds])
        assert (got == want).all(), "depth %d" % depth
        assert slow == sum(depth > k for k in accepted), "depth %d" % depth


@pytest.mark.parametrize("size", (2, 3))
def test_emulated_draws_equal_numpy(emul, size):
    a = 12 if size == 3 else 6
    rng = np.random.RandomState(20 + size)
    seeds = np.concatenate([EDGE_SEEDS, rng.randint(0, 2 ** 32, size=3000, dtype=np.uint64)]).astype(np.int64)
    want = np.stack([np.random.RandomState(int(s)).randint(a, size=128) for s in seeds])
    accepted = np.array([_accepted_in_fast_draws(size, int(s)) for s in seeds])
    for depth in DEPTHS:
        got, slow = _draw(emul, size, seeds, depth)
        assert (got == want[:, :depth]).all(), "depth %d" % depth
        assert slow == int((depth > accepted).sum())
