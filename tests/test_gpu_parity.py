"""GPU parity tests: the CUDA path, called through the C ABI, against the oracle and the
golden vectors generated from the reference.  Bit-exact everywhere (integer / byte work).
Run on the B200 box:  python -m pytest tests -m gpu -x -q
"""
import copy
import os
import ctypes

import numpy as np
import pytest
import torch

import rubiks_cube_solver_b200 as R
from rubiks_cube_solver_b200 import _lib, adi, ops

from oracle import cube_c as C
from oracle import cube_np as O
from oracle import tables as T
from oracle.gen_golden import ExactValueNet

from conftest import golden

pytestmark = pytest.mark.gpu
SIZES = (2, 3)
ONE = {torch.bfloat16: 1.0, torch.float32: 1.0, torch.uint8: 1}


def dev():
    return torch.device("cuda", 0)


def cu(a, dtype=np.uint8):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=dtype)).to(dev())


def onehot_to_u8(t):
    return (t.float() == 1.0).to(torch.uint8).cpu().numpy(), bool(((t.float() == 0) | (t.float() == 1)).all())


# ------------------------------------------------------------------ golden vectors (reference)
@pytest.mark.parametrize("size", SIZES)
def test_config1_golden(size):
    g = golden("config1_%d.npz" % size)
    counters = ops.new_counters(dev())
    states, solved, reward = ops.scramble(size, cu(g["moves"]), counters=counters)
    assert (states.cpu().numpy() == g["stickers"]).all()
    assert (solved.cpu().numpy().astype(bool) == g["done"]).all()
    assert (reward.cpu().numpy() == g["reward"]).all()
    assert counters.tolist()[:2] == [int(g["done"].sum()), 1024]
    for dt in (torch.uint8, torch.float32, torch.bfloat16):
        enc, clean = onehot_to_u8(ops.encode(size, states, dtype=dt))
        assert clean and (enc == g["onehot"]).all(), dt
    # bf16 1.0 must be the exact bit pattern the net reads
    raw = ops.encode(size, states, dtype=torch.bfloat16).view(torch.int16).cpu().numpy()
    assert set(np.unique(raw)) == {0, 0x3f80}


@pytest.mark.parametrize("size", SIZES)
def test_walks_golden_step_by_step(size):
    g = golden("walks_%d.npz" % size)
    n, d = g["moves"].shape
    states = ops.solved_states(size, n, dev())
    assert (states.cpu().numpy() == O.solved_states(size, n)).all()
    for k in range(d):
        states, solved, reward = ops.step(size, states, cu(g["moves"][:, k]))
        assert (states.cpu().numpy() == g["stickers"][:, k]).all(), k
        assert (solved.cpu().numpy().astype(bool) == g["done"][:, k]).all()
        assert (reward.cpu().numpy() == g["reward"][:, k]).all()
        enc, _ = onehot_to_u8(ops.encode(size, states, dtype=torch.uint8))
        assert (enc == g["onehot"][:, k]).all()
    assert g["done"].any()


@pytest.mark.parametrize("size", SIZES)
def test_expand_golden(size):
    g = golden("expand_%d.npz" % size)
    res = ops.expand(size, cu(g["parents"]), dtype=torch.bfloat16, want_children=True, want_parent_onehot=True)
    assert (res["children"].cpu().numpy() == g["children"]).all()
    assert (res["solved"].cpu().numpy().astype(bool) == g["child_solved"]).all()
    assert (res["reward"].cpu().numpy() == np.where(g["child_solved"], 1.0, -1.0)).all()
    enc, clean = onehot_to_u8(res["child_onehot"])
    assert clean and (enc == g["child_onehot"]).all()
    enc, _ = onehot_to_u8(res["parent_onehot"])
    assert (enc == O.encode(size, g["parents"])).all()


def test_decode_golden():
    g = golden("decode_2.npz")
    for dt in (torch.uint8, torch.float32, torch.bfloat16):
        got = ops.decode(2, cu(g["onehot"]).to(dt).contiguous())
        assert (got.cpu().numpy() == g["stickers"]).all()
    with pytest.raises(NotImplementedError):
        ops.decode(3, cu(np.zeros((1, 20, 24))))


# ------------------------------------------------------------------ oracle, seeded inputs
@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("depth", (0, 1, 3, 4, 7, 8, 9, 20, 30, 31, 32, 61, 100, 128, 129, 200, 255, 320, 321, 400))
def test_scramble_vs_oracle_depths(size, depth):
    rng = np.random.RandomState(depth + 100 * size)
    n = 3000
    moves = rng.randint(T.N_ACTIONS[size], size=(n, depth)).astype(np.uint8)
    if depth >= 2:
        h = depth // 2
        moves[:64, h:2 * h] = moves[:64, :h][:, ::-1] ^ 1
        if depth % 2:
            moves[:64, -1] = 12                                    # no-op row keeps them solved
    counters = ops.new_counters(dev())
    states, solved, reward = ops.scramble(size, cu(moves), counters=counters)
    if depth >= 2 and depth % 2:
        # the first 64 rows end with the no-op index: the oracle applies their first depth-1 moves
        want, want_solved, want_reward, _ = C.scramble(size, np.where(moves == 12, 0, moves))
        want[:64], want_solved[:64], want_reward[:64], _ = C.scramble(size, moves[:64, :-1])
        cnt = int(want_solved.sum())
    else:
        want, want_solved, want_reward, cnt = C.scramble(size, moves)
    assert (states.cpu().numpy() == want).all()
    assert (solved.cpu().numpy().astype(bool) == want_solved).all()
    assert (reward.cpu().numpy() == want_reward).all()
    assert counters.tolist()[:2] == [cnt, n]
    if depth >= 2:
        assert solved[:64].all()


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("depth", (8, 16, 24, 32, 48, 64, 72, 96, 128, 200, 320))
def test_scramble_swizzled_move_tiles(size, depth):
    """Depths whose flat tile image bank-conflicts stage K1p's move tiles by a 2-D tensor copy with the
    128-byte swizzle.  Several tiles per warp, so both move buffers and their barriers' phases are reused;
    a ragged tail; rows that come back to solved."""
    rng = np.random.RandomState(depth + 1000 * size)
    n = 148 * (32 if depth <= 96 else 8) * 64 * 3 + 77
    moves = rng.randint(T.N_ACTIONS[size], size=(n, depth)).astype(np.uint8)
    h = depth // 2
    back = rng.choice(n, 500, replace=False)
    moves[back, h:] = moves[back, :h][:, ::-1] ^ 1
    counters = ops.new_counters(dev())
    states, solved, reward = ops.scramble(size, cu(moves), counters=counters)
    want, want_solved, want_reward, cnt = C.scramble(size, moves)
    assert (states.cpu().numpy() == want).all()
    assert (solved.cpu().numpy().astype(bool) == want_solved).all()
    assert (reward.cpu().numpy() == want_reward).all()
    assert counters.tolist()[:2] == [cnt, n] and want_solved[back].all()


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("n", (1, 2, 255, 256, 257, 513, 100003))
def test_scramble_ragged_sizes(size, n):
    rng = np.random.RandomState(n)
    depth = 20 if size == 2 else 30
    moves = rng.randint(T.N_ACTIONS[size], size=(n, depth)).astype(np.uint8)
    states, solved, _ = ops.scramble(size, cu(moves))
    want, ws, _, _ = C.scramble(size, moves)
    assert (states.cpu().numpy() == want).all() and (solved.cpu().numpy().astype(bool) == ws).all()


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("n,depth", [(n, d) for n in (63, 64, 65, 129) for d in (2, 95, 96, 97, 319, 320, 321)]
                         + [(n, d) for n in (127, 128, 191, 257) for d in (1, 20, 30, 31, 32, 33)]
                         + [(64 * 148 * 24 + 1, 30), (64 * 148 * 32 + 65, 20), (128 * 148 * 20 * 3 + 127, 20)])
def test_scramble_tile_and_depth_boundaries(size, n, depth):
    """K1p handles whole tiles (64 rows; 128 for shallow 2x2x2 sequences, four instances per lane) at depth
    1..320; the single-move kernels take the ragged tail, deeper sequences and everything around: the
    seams must not show."""
    rng = np.random.RandomState(n % 1000 + depth)
    moves = rng.randint(T.N_ACTIONS[size], size=(n, depth)).astype(np.uint8)
    if depth % 2 == 0:
        moves[-3:, depth // 2:] = moves[-3:, :depth // 2][:, ::-1] ^ 1                   # the last rows end solved
    counters = ops.new_counters(dev())
    states, solved, reward = ops.scramble(size, cu(moves), counters=counters)
    want, ws, wr, cnt = C.scramble(size, moves)
    assert (states.cpu().numpy() == want).all()
    assert (solved.cpu().numpy().astype(bool) == ws).all() and (depth % 2 or ws[-3:].all())
    assert (reward.cpu().numpy() == wr).all()
    assert counters.tolist()[:2] == [cnt, n]


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("n", (63, 64, 65, 4097))
@pytest.mark.parametrize("depth", (1, 64, 65))
def test_walk_tile_and_depth_boundaries(size, n, depth):
    """K2p (lane-private layout) handles whole 64-row tiles at depth 1..64, walk_tile_kernel the rest."""
    rng = np.random.RandomState(n + depth)
    A = T.N_ACTIONS[size]
    start = O.scramble(size, rng.randint(A, size=(n, 7)))
    moves = rng.randint(A, size=(n, depth)).astype(np.uint8)
    counters = ops.new_counters(dev())
    out, solved, reward = ops.walk(size, cu(start), cu(moves), counters=counters)
    want = O.scramble(size, moves, init=start)
    ws = O.is_solved(size, want)
    assert (out.cpu().numpy() == want).all() and (solved.cpu().numpy().astype(bool) == ws).all()
    assert (reward.cpu().numpy() == O.rewards(ws)).all()
    assert counters.tolist()[:2] == [int(ws.sum()), n]


@pytest.mark.parametrize("depth", (30, 32))
def test_persistent_kernels_on_concurrent_streams_and_in_a_graph(depth):
    """The tile scheduler's counters come from a ring of slots that every kernel re-arms: launches that
    overlap on different streams must not see each other, and a captured launch must replay (depth 32:
    the swizzled variant, whose tensor map of the move array is a kernel parameter baked into the graph)."""
    rng = np.random.RandomState(9)
    n = 64 * 600 + 5
    streams = [torch.cuda.Stream() for _ in range(4)]
    jobs = []
    for i, st in enumerate(streams * 3):
        moves = rng.randint(12, size=(n, depth)).astype(np.uint8)
        m = cu(moves)
        torch.cuda.synchronize()
        with torch.cuda.stream(st):
            states, solved, _ = ops.scramble(3, m)
            stepped, s2, _ = ops.step(3, states.clone(), m[:, 0].contiguous())
        jobs.append((moves, states, stepped))
    torch.cuda.synchronize()
    for moves, states, stepped in jobs:
        want = O.scramble(3, moves)
        assert (states.cpu().numpy() == want).all()
        assert (stepped.cpu().numpy() == O.apply_moves(3, want, moves[:, 0])).all()
    # CUDA graph: capture one scramble, replay it with new moves in the same buffer
    moves = cu(rng.randint(12, size=(n, depth)).astype(np.uint8))
    out = torch.empty((n, 54), dtype=torch.uint8, device=dev())
    so = torch.empty(n, dtype=torch.uint8, device=dev())
    rw = torch.empty(n, dtype=torch.float32, device=dev())
    ops.scramble(3, moves, out=out, solved=so, reward=rw)              # warm-up outside the capture
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        ops.scramble(3, moves, out=out, solved=so, reward=rw)
    for _ in range(3):
        fresh = rng.randint(12, size=(n, depth)).astype(np.uint8)
        moves.copy_(torch.from_numpy(fresh))
        g.replay()
        torch.cuda.synchronize()
        assert (out.cpu().numpy() == O.scramble(3, fresh)).all()


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("depth", (1, 10, 30, 100, 128))
def test_moves_from_seeds_equal_numpy_legacy_randint(size, depth):
    """K0 (cube_moves_from_seeds): the device's MT19937 + masked rejection against
    np.random.RandomState(seed).randint(A, size=depth), the draw of reset(seed, k) (cube_env.py:62-65)."""
    A = T.N_ACTIONS[size]
    seeds = list(range(0, 1500)) + [10 * i for i in range(200)] + [2 ** 31 - 1, 2 ** 31, 2 ** 32 - 1, 123456789]
    got = ops.moves_from_seeds(size, seeds, depth).cpu().numpy()
    for i, sd in enumerate(seeds):
        assert (got[i] == np.random.RandomState(sd).randint(A, size=depth)).all(), sd
    with pytest.raises(ValueError):
        ops.moves_from_seeds(size, [2 ** 32], depth)


def test_batched_reset_from_seeds_matches_config1_golden():
    """BatchedCubeEnv.reset(seeds=...) draws its moves on the device: config 1 end to end on the GPU."""
    from rubiks_cube_solver_b200 import rollout
    for size in SIZES:
        g = golden("config1_%d.npz" % size)
        env = R.BatchedCubeEnv(1024, cube_size=size, obs_dtype=torch.float32)
        obs, reward, done = env.reset(seeds=range(1024), scramble_count=10)
        assert (env.sim_cube.cpu().numpy() == g["stickers"]).all()
        assert (obs.cpu().numpy() == g["onehot"]).all()
        assert (done.cpu().numpy().astype(bool) == g["done"]).all()
        host = rollout.reference_scrambles(size, [0, 10, 20], [1, 5, 30])
        devm = rollout.reference_scrambles_device(size, [0, 10, 20], [1, 5, 30]).cpu().numpy()
        assert (host == devm).all()


def test_scramble_empty_and_optional_outputs():
    for size in SIZES:
        s, so, rw = ops.scramble(size, torch.empty((0, 5), dtype=torch.uint8, device=dev()))
        assert s.shape == (0, T.N_STICKERS[size]) and so.numel() == 0
        moves = cu(np.random.RandomState(1).randint(T.N_ACTIONS[size], size=(300, 6)))
        s2, so2, rw2 = ops.scramble(size, moves, want_flags=False)
        assert so2 is None and rw2 is None
        assert (s2.cpu().numpy() == O.scramble(size, moves.cpu().numpy())).all()


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("depth", (1, 2, 7))
def test_walk_vs_oracle_any_bytes(size, depth):
    rng = np.random.RandomState(5 + depth)
    n = 5000
    A, S = T.N_ACTIONS[size], T.N_STICKERS[size]
    start = O.scramble(size, rng.randint(A, size=(n, 11)))
    start[:100] = rng.randint(0, 256, size=(100, S))               # the gather is defined for any bytes
    moves = rng.randint(A, size=(n, depth)).astype(np.uint8)
    start[100:200] = O.scramble(size, moves[100:200, ::-1] ^ 1)
    out, solved, reward = ops.walk(size, cu(start), cu(moves))
    want = O.scramble(size, moves, init=start)
    assert (out.cpu().numpy() == want).all()
    assert (solved.cpu().numpy().astype(bool) == O.is_solved(size, want)).all()
    assert solved[100:200].all()
    # in place
    st = cu(start)
    ops.walk(size, st, cu(moves), out=st)
    assert (st.cpu().numpy() == want).all()
    sol2, rew2 = ops.is_solved(size, st)
    assert (sol2.cpu().numpy().astype(bool) == O.is_solved(size, want)).all()
    assert (rew2.cpu().numpy() == O.rewards(O.is_solved(size, want))).all()


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("dtype", (torch.bfloat16, torch.float32, torch.uint8))
@pytest.mark.parametrize("n", (1, 5, 16, 37, 4099))
def test_expand_vs_oracle(size, dtype, n):
    rng = np.random.RandomState(n)
    A, S = T.N_ACTIONS[size], T.N_STICKERS[size]
    parents = O.scramble(size, rng.randint(A, size=(n, 9)))
    parents[0] = O.scramble(size, np.array([[3]]))[0]
    counters = ops.new_counters(dev())
    res = ops.expand(size, cu(parents), dtype=dtype, want_children=True, want_parent_onehot=True, counters=counters)
    want_c, want_s = O.expand(size, parents)
    assert (res["children"].cpu().numpy() == want_c).all()
    assert (res["solved"].cpu().numpy().astype(bool) == want_s).all() and res["solved"][0, 2] == 1
    assert counters.tolist()[:2] == [int(want_s.sum()), n * A]
    enc, clean = onehot_to_u8(res["child_onehot"])
    assert clean and (enc.reshape(n * A, -1) == O.encode(size, want_c.reshape(n * A, S)).reshape(n * A, -1)).all()
    enc, clean = onehot_to_u8(res["parent_onehot"])
    assert clean and (enc == O.encode(size, parents)).all()
    # expand[a] == step(a)
    for a in (0, A - 1):
        stepped, _, _ = ops.step(size, cu(parents), torch.full((n,), a, dtype=torch.uint8, device=dev()))
        assert (stepped == res["children"][:, a]).all()


@pytest.mark.parametrize("dtype", (torch.bfloat16, torch.float32, torch.uint8))
@pytest.mark.parametrize("n", (1, 63, 64, 128, 129, 1000, 70001))
@pytest.mark.parametrize("want_children,want_parent", ((True, True), (True, False), (False, True)))
def test_leaf_expand_vs_oracle(dtype, n, want_children, want_parent):
    # the MCTS-leaf shape of cube_expand for 2x2x2 (register-resident kernel + generic remainder)
    rng = np.random.RandomState(n)
    parents = O.scramble(2, rng.randint(6, size=(n, 9)))
    parents[0] = O.scramble(2, np.array([[3]]))[0]
    if n > 1:
        parents[n // 2] = O.solved_states(2, 1)[0]
    counters = ops.new_counters(dev())
    res = ops.expand(2, cu(parents), dtype=dtype, want_children=want_children, want_child_onehot=False,
                     want_parent_onehot=want_parent, counters=counters)
    want_c, want_s = O.expand(2, parents)
    assert res["child_onehot"] is None
    assert (res["solved"].cpu().numpy().astype(bool) == want_s).all() and res["solved"][0, 2] == 1
    assert (res["reward"].cpu().numpy() == np.where(want_s, 1.0, -1.0)).all()
    assert counters.tolist()[:2] == [int(want_s.sum()), n * 6]
    if want_children:
        assert (res["children"].cpu().numpy() == want_c).all()
    if want_parent:
        enc, clean = onehot_to_u8(res["parent_onehot"])
        assert clean and (enc == O.encode(2, parents)).all()


def test_validate_actions_and_errors():
    good = cu(np.random.RandomState(0).randint(12, size=(1000, 30)))
    ops.validate_actions(3, good)
    with pytest.raises(IndexError):
        ops.validate_actions(2, good)                               # 6..11 are out of range for 2x2x2
    bad = good.clone()
    bad[777, 3] = 12
    with pytest.raises(IndexError):
        ops.validate_actions(3, bad)
    bad[777, 3] = 200
    with pytest.raises(IndexError):
        ops.validate_actions(3, bad)
    with pytest.raises(NotImplementedError):
        ops.scramble(4, good)
    with pytest.raises(TypeError):
        ops.scramble(3, good.cpu())
    with pytest.raises(ValueError):                                 # mis-aligned device pointer
        lib = _lib.load()
        raw = torch.empty(4096, dtype=torch.uint8, device=dev())
        _lib.check(lib.cube_scramble(3, ctypes.c_void_p(raw.data_ptr() + 1), 8, 4, ctypes.c_void_p(raw.data_ptr() + 1024),
                                     None, None, None, None), "cube_scramble")


# ------------------------------------------------------------------ full-size properties (BASELINE configs 2, 3)
@pytest.mark.parametrize("size,n,depth", ((2, 16 * 2 ** 20, 20), (3, 8 * 2 ** 20, 30)))
def test_full_size_properties(size, n, depth):
    A = T.N_ACTIONS[size]
    gen = torch.Generator(device=dev()).manual_seed(1234)
    moves = torch.randint(0, A, (n, depth), dtype=torch.uint8, device=dev(), generator=gen)
    counters = ops.new_counters(dev())
    states, solved, reward = ops.scramble(size, moves, counters=counters)
    # sampled replay through the oracle: first 4096 rows, 4096 random rows, and the solved count of 1 Mi rows
    idx = np.concatenate((np.arange(4096), np.random.RandomState(7).randint(n, size=4096)))
    want, ws, wr, _ = C.scramble(size, moves[idx].cpu().numpy())
    assert (states[idx].cpu().numpy() == want).all()
    assert (solved[idx].cpu().numpy().astype(bool) == ws).all() and (reward[idx].cpu().numpy() == wr).all()
    sub = slice(n // 2, n // 2 + 2 ** 20)
    _, ws, _, cnt = C.scramble(size, moves[sub].cpu().numpy())
    assert int(solved[sub].sum()) == cnt
    assert int(counters[0]) == int(solved.sum()) and int(counters[1]) == n
    assert float(reward.double().sum()) == 2 * int(counters[0]) - n
    # every sticker row is a permutation of the solved multiset (checksum of checksums)
    per = T.N_STICKERS[size] // 6
    hist = torch.stack([(states == c).sum(dim=1) for c in range(6)], dim=1)
    assert bool((hist == per).all())
    # scramble followed by its inverse is the identity: all N instances solved
    undo = torch.cat((moves, moves.flip(1) ^ 1), dim=1).contiguous()
    counters.zero_()
    s2, so2, _ = ops.scramble(size, undo, counters=counters)
    assert int(counters[0]) == n and bool(so2.all())
    assert bool((s2 == ops.solved_states(size, 1, dev())).all())
    # one more step on the resident states equals a depth+1 scramble
    extra = torch.randint(0, A, (n,), dtype=torch.uint8, device=dev(), generator=gen)
    stepped, so3, _ = ops.step(size, states.clone(), extra)
    longer, so4, _ = ops.scramble(size, torch.cat((moves, extra[:, None]), dim=1).contiguous())
    assert bool((stepped == longer).all()) and bool((so3 == so4).all())


def test_config4_and_5_shapes_sampled():
    # config 4 (3x3x3 ADI batch) and config 5 (2x2x2 MCTS leaves) on a slice, vs the oracle
    gen = torch.Generator(device=dev()).manual_seed(99)
    moves = torch.randint(0, 12, (4096, 30), dtype=torch.uint8, device=dev(), generator=gen)
    trail = adi.scramble_prefixes(3, moves)                           # [cube, depth, S]: cube-major, one launch
    _, want_trail, _ = O.scramble(3, moves.cpu().numpy(), per_step=True)
    assert (trail.cpu().numpy() == want_trail).all()
    parents = trail.view(-1, 54)
    res = ops.expand(3, parents, dtype=torch.bfloat16)
    sample = np.random.RandomState(0).randint(parents.shape[0], size=2048)
    pc, ps = O.expand(3, parents[sample].cpu().numpy())
    enc, clean = onehot_to_u8(res["child_onehot"][sample])
    assert clean and (enc.reshape(2048 * 12, 480) == O.encode(3, pc.reshape(-1, 54)).reshape(-1, 480)).all()
    assert (res["solved"][sample].cpu().numpy().astype(bool) == ps).all()
    leaves_moves = torch.randint(0, 6, (2 ** 16, 11), dtype=torch.uint8, device=dev(), generator=gen)
    leaves, _, _ = ops.scramble(2, leaves_moves)
    res = ops.expand(2, leaves, dtype=torch.bfloat16, want_children=True, want_child_onehot=False,
                     want_parent_onehot=True)
    lc, ls = O.expand(2, leaves.cpu().numpy())
    assert (res["children"].cpu().numpy() == lc).all() and (res["solved"].cpu().numpy().astype(bool) == ls).all()
    enc, _ = onehot_to_u8(res["parent_onehot"])
    assert (enc == O.encode(2, leaves.cpu().numpy())).all()


def test_host_pipeline_matches_device_path():
    for size, depth in ((3, 30), (2, 20)):
        n = 300000 + 77
        moves = torch.from_numpy(np.random.RandomState(size).randint(T.N_ACTIONS[size], size=(n, depth))
                                 .astype(np.uint8)).pin_memory()
        pipe = ops.HostScramblePipeline(size, depth, chunk_instances=1 << 16, n_stages=3)
        states, solved, reward, count = pipe.run(moves)
        want, ws, wr, cnt = C.scramble(size, moves.numpy())
        assert (states.numpy() == want).all() and (solved.numpy().astype(bool) == ws).all()
        assert (reward.numpy() == wr).all() and count == cnt
        states2, _, _, count2 = pipe.run(moves[:1000].contiguous())          # reusable, ragged
        assert (states2.numpy() == want[:1000]).all() and count2 == int(ws[:1000].sum())
        pipe.close()


# ------------------------------------------------------------------ the drop-in env
@pytest.mark.parametrize("size", SIZES)
def test_cube_env_drop_in(size):
    g = golden("config1_%d.npz" % size)
    w = golden("walks_%d.npz" % size)
    env = R.make_env(torch.device("cpu"), size)
    assert env.state_dim == list(T.STATE_DIM[size]) and env.action_dim == T.N_ACTIONS[size]
    assert env.action_to_sim_action[size] == T.ACTIONS[size]
    assert env.sim_cube.dtype == np.int64 and (env.sim_cube == T.SOLVED[size]).all()
    before = np.random.get_state()[1].copy()
    for seed in (0, 1, 500, 1023):
        obs = env.reset(seed=seed, scramble_count=10)
        assert obs.dtype == np.dtype(str(g["obs_dtype"])) and obs.shape == tuple(T.STATE_DIM[size])
        assert (env.sim_cube == g["stickers"][seed]).all() and (obs == g["onehot"][seed]).all()
        assert obs is env.cube
    assert (np.random.get_state()[1] == before).all()
    with pytest.raises(UnboundLocalError):
        env.reset(seed=0, scramble_count=0)
    env.init_state()                                                  # step before any reset (train.py:155 path)
    for k, a in enumerate(w["moves"][0]):
        obs, r, d, info = env.step(int(a))
        assert (obs == w["onehot"][0, k]).all() and (env.sim_cube == w["stickers"][0, k]).all()
        assert isinstance(r, float) and r == w["reward"][0, k] and isinstance(d, bool) and d == w["done"][0, k]
        assert info == {}
    with pytest.raises(IndexError):
        env.step(T.N_ACTIONS[size])
    # deepcopy independence (mcts.py:37,96,101)
    env.reset(seed=3, scramble_count=5)
    twin = copy.deepcopy(env)
    twin.step(0)
    assert not (twin.sim_cube == env.sim_cube).all()
    env.step(0)
    assert (twin.sim_cube == env.sim_cube).all() and (twin.cube == env.cube).all()
    # undo -> reward +1, done
    env.init_state()
    seq = [1, 4, 2]
    for a in seq:
        env.step(a)
    for a in reversed(seq[1:]):
        _, r, d, _ = env.step(a ^ 1)
        assert r == -1.0 and not d
    _, r, d, _ = env.step(seq[0] ^ 1)
    assert r == 1.0 and d is True
    with pytest.raises(NotImplementedError):
        R.make_env(torch.device("cpu"), 4)
    if size == 2:
        d2 = golden("decode_2.npz")
        assert (env.state_to_sim_state(d2["onehot"][0].astype(np.float64)) == d2["stickers"][0]).all()
    else:
        with pytest.raises(NotImplementedError):
            env.state_to_sim_state(env.cube)


@pytest.mark.parametrize("size", SIZES)
def test_adi_against_reference_golden(size):
    g = golden("adi_%d.npz" % size)
    n, d = g["moves"].shape
    net = ExactValueNet(T.STATE_DIM[size], T.N_ACTIONS[size])
    env = R.make_env(torch.device("cpu"), size)
    buf = []
    saved = np.random.get_state()
    np.random.seed(11)
    env.get_random_samples(buf, net, d, n, float(g["temperature"]))
    after = np.random.get_state()[1].copy()
    np.random.set_state(saved)
    assert len(buf) == n * d
    assert (np.array([b["state"] for b in buf]) == g["state"]).all()
    assert buf[0]["state"].dtype == (np.float64 if size == 2 else np.int64)
    assert [b["target_policy"] for b in buf] == list(g["target_policy"])
    assert [b["target_value"] for b in buf] == list(g["target_value"])
    assert [b["scramble_count"] for b in buf] == list(g["scramble_count"])
    assert np.array_equal(np.array([b["error"] for b in buf]), g["error"])
    # the global RNG advanced exactly as the reference's loop advances it
    ref = np.random.RandomState(11)
    ref.randint(T.N_ACTIONS[size], size=(n, d))
    assert (ref.get_state()[1] == after).all()
    # get_target_value on single cubes, including the first-solved-child override
    env.init_state()
    env.step(5)
    tv, tp, err = env.get_target_value(net, 1, 1.0)
    assert (tv, tp) == (1.0, 4)
    k = 0
    env.init_state()
    for a in g["moves"][0]:
        env.step(int(a))
        tv, tp, err = env.get_target_value(net, k + 1, float(g["temperature"]))
        assert tv == g["target_value"][k] and tp == g["target_policy"][k] and err == g["error"][k]
        k += 1


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("temperature", (1.0, 0.5, 0.3))
def test_adi_targets_kernel_vs_reference_rules(size, temperature):
    """K4 (cube_adi_targets) against the reference's rules restated per parent in Python:
    first solved child -> (1.0, a); else torch.max of float32 V(child) + (-1.0), first maximum wins
    (cube_env.py:217-220, 243-245); error = |V(s) - target| * k ** (-T) in Python floats (:247-251)."""
    rng = np.random.RandomState(5 + size)
    a, p = T.N_ACTIONS[size], 5000
    cv = rng.randn(p, a).astype(np.float32)
    cv[:500] = np.round(cv[:500])                                    # ties: the first maximum must win
    solved = (rng.rand(p, a) < 0.03).astype(np.uint8)
    solved[1000:1010] = 1
    pv = rng.randn(p).astype(np.float32)
    k = rng.randint(1, 31, size=p).astype(np.int32)
    tv, tp, err = ops.adi_targets(size, torch.from_numpy(cv).to(dev()), torch.from_numpy(solved).to(dev()),
                                  torch.from_numpy(pv).to(dev()), torch.from_numpy(k).to(dev()), temperature)
    tv, tp, err = tv.cpu().numpy(), tp.cpu().numpy(), err.cpu().numpy()
    assert tv.dtype == np.float32 and tp.dtype == np.int64 and err.dtype == np.float64
    for i in range(p):
        if solved[i].any():
            want_v, want_p = 1.0, int(solved[i].argmax())
        else:
            value = torch.from_numpy(cv[i]) + torch.full((a,), -1.0)
            m, j = torch.max(value, -1, keepdim=True)
            want_v, want_p = m.item(), j.item()
        want_e = abs(float(pv[i]) - want_v) * int(k[i]) ** (-1 * temperature)
        assert float(tv[i]) == want_v and int(tp[i]) == want_p and float(err[i]) == want_e, i


def test_batched_env_matches_reference_seeds():
    for size in SIZES:
        g = golden("config1_%d.npz" % size)
        env = R.BatchedCubeEnv(1024, cube_size=size, obs_dtype=torch.float32)
        obs, reward, done = env.reset(seeds=range(1024), scramble_count=10)
        assert (env.sim_cube.cpu().numpy() == g["stickers"]).all()
        assert (obs.cpu().numpy() == g["onehot"]).all()
        assert (done.cpu().numpy().astype(bool) == g["done"]).all() and (reward.cpu().numpy() == g["reward"]).all()
        act = torch.from_numpy(g["moves"][:, -1] ^ 1)
        obs, reward, done, info = env.step(act, validate=True)
        want = O.scramble(size, g["moves"][:, :-1])
        assert (env.sim_cube.cpu().numpy() == want).all() and info == {}
        assert (obs.cpu().numpy() == O.encode(size, want)).all()


class ExactPolicyNet(torch.nn.Module):
    """DeepCube-shaped net (model.py:31-45) whose outputs are exact in fp32 on any device."""

    def __init__(self, state_dim, action_dim, seed=3):
        super().__init__()
        r = np.random.RandomState(seed)
        d = state_dim[0] * state_dim[1]
        self.w = torch.nn.Parameter(torch.tensor(r.randint(-512, 513, size=(d, action_dim)).astype(np.float32) / 1024.0),
                                    requires_grad=False)

    def forward(self, x):
        if x.dim() == 2:
            x = x.unsqueeze(0)
        logits = x.reshape(x.shape[0], -1).float() @ self.w
        return logits.sum(dim=1, keepdim=True), logits


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("mask", (False, True))
def test_greedy_rollout_matches_scalar_env(size, mask):
    from rubiks_cube_solver_b200 import rollout
    from oracle.scalar_env import ScalarCubeEnv
    net = ExactPolicyNet(T.STATE_DIM[size], T.N_ACTIONS[size])
    seeds, depths, horizon = [0, 10, 20, 30], [1, 2, 3, 5], 12
    moves = rollout.reference_scrambles(size, seeds, depths)
    res = rollout.greedy_solve(net.to(dev()), size, moves, max_timesteps=horizon, mask_inverse=mask)
    env = ScalarCubeEnv(size)
    cpu_net = ExactPolicyNet(T.STATE_DIM[size], T.N_ACTIONS[size])
    k = 0
    for d in depths:
        for s in seeds:
            state = env.reset(seed=s, scramble_count=d)
            first, pre = 0, None
            for t in range(1, horizon + 1):
                _, logits = cpu_net(torch.tensor(state).float())
                order = logits[0].argsort(descending=True, stable=True)
                a = int(order[0])
                if mask and pre is not None and a == (pre ^ 1):
                    a = int(order[1])
                state, _, done, _ = env.step(a)
                pre = a
                if done:
                    first = t
                    break
            assert int(res["steps"][k]) == first and bool(res["solved"][k]) == (first > 0), (d, s)
            if first == 0:
                assert (res["states"][k].cpu().numpy() == env.sim_cube).all()
            k += 1
    pct = rollout.validation(net.to(dev()), size, sample_scramble_count=3, sample_cube_count=4, max_timesteps=6)
    assert len(pct) == 3 and all(0.0 <= p <= 100.0 for p in pct)


@pytest.mark.parametrize("size", SIZES)
def test_mcts_leaf_batch_matches_per_leaf_expand(size):
    # MCTS.expand (mcts.py:83-113) per leaf with the scalar env vs one batched call
    import copy as _copy
    from rubiks_cube_solver_b200 import mcts_batch
    from oracle.scalar_env import ScalarCubeEnv
    net = ExactPolicyNet(T.STATE_DIM[size], T.N_ACTIONS[size])
    rng = np.random.RandomState(4)
    A = T.N_ACTIONS[size]
    n = 200
    leaves = O.scramble(size, rng.randint(A, size=(n, 6)))
    leaves[0] = O.scramble(size, np.array([[2]]))[0]
    out = mcts_batch.expand_leaves(net.to(dev()), size, cu(leaves), obs_dtype=torch.float32)
    cpu_net = ExactPolicyNet(T.STATE_DIM[size], T.N_ACTIONS[size])
    env = ScalarCubeEnv(size)
    for i in range(0, n, 7):
        env.sim_cube = leaves[i].astype(np.int64)
        env.cube = env._observe(env.sim_cube)
        value, logits = cpu_net(torch.tensor(env.cube).float())
        policy = torch.nn.functional.softmax(logits, dim=-1)[0]
        assert float(out["value"][i]) == float(value[0, 0])
        assert torch.allclose(out["policy"][i].cpu(), policy, atol=1e-6)
        for a in range(A):
            child = _copy.deepcopy(env)
            _, _, done, _ = child.step(a)
            assert (out["children"][i, a].cpu().numpy() == child.sim_cube).all() and bool(out["done"][i, a]) == done
    assert bool(out["done"][0, 3])


@pytest.mark.parametrize("size", SIZES)
def test_batched_mcts_matches_reference_golden(size):
    """BatchedMCTS (device tree store, all cubes in lock-step) against the reference's own mcts.py run
    on its own env (tests/golden/mcts_*.npz, oracle/gen_golden.py): returned action lists, simulations
    used, node counts and the root's N / W / L after the search."""
    from rubiks_cube_solver_b200 import mcts_batch
    from oracle.gen_golden import ExactSearchNet, MCTS_CFG
    g = golden("mcts_%d.npz" % size)
    cases = g["cases"]
    roots = np.stack([O.scramble(size, O.reference_moves(size, int(sd), int(d))[None])[0] for sd, d in cases])
    net = ExactSearchNet(T.STATE_DIM[size], T.N_ACTIONS[size]).to(dev())
    cfg = MCTS_CFG["mcts"]
    search = mcts_batch.BatchedMCTS(net, size, num_sim=cfg["numMCTSSim"], cpuct=cfg["cpuct"],
                                    virtual_loss_const=cfg["virtual_loss_const"], value_min=cfg["value_min"])
    out = search.run(cu(roots), seeds=[1000 + int(sd) for sd, _ in cases])
    assert (out["n_sims"].cpu().numpy() == g["n_sims"]).all()
    assert (out["n_actions"].cpu().numpy() == g["n_actions"]).all()
    assert (out["actions"].cpu().numpy() == g["actions"]).all()
    assert (out["n_nodes"].cpu().numpy() == g["n_nodes"]).all()
    assert (out["root_N"].cpu().numpy() == g["root_N"]).all()
    assert (out["root_L"].cpu().numpy() == g["root_L"]).all()
    assert (out["root_W"].cpu().numpy().astype(np.float64) == g["root_W"]).all()
    assert out["solved"].any() and not out["solved"].all()


@pytest.mark.parametrize("size,consts", [pytest.param(2, None, id="2"), pytest.param(3, None, id="3")] + [
    pytest.param(size, consts, id="%d-cpuct%g-vl%d-vmin%g-cap%d" % ((size,) + consts))
    for size in SIZES for consts in ((0.37, 160, -3.5, 105), (2.5, 1000, 0.25, 107))])
def test_batched_mcts_matches_oracle_more_cases(size, consts):
    """More cubes, fewer simulations, against oracle/mcts_ref.py (itself pinned to the reference by
    tests/test_oracle.py): ragged batch sizes and cubes solved at different simulations.  `consts` =
    (cpuct, virtual_loss_const, value_min, path_cap) other than the defaults, the path_cap not a multiple of 4."""
    import random
    from rubiks_cube_solver_b200 import mcts_batch
    from oracle import mcts_ref
    from oracle.gen_golden import ExactSearchNet
    from oracle.scalar_env import ScalarCubeEnv
    n, num_sim = 70, 12
    rng = np.random.RandomState(17 + size)
    A = T.N_ACTIONS[size]
    depths = rng.randint(1, 4, size=n)
    roots = np.stack([O.scramble(size, rng.randint(A, size=(1, int(d))))[0] for d in depths])
    gpu_net = ExactSearchNet(T.STATE_DIM[size], A).to(dev())
    cpu_net = ExactSearchNet(T.STATE_DIM[size], A)
    kw, search_kw = {}, {}
    if consts is not None:
        kw = dict(cpuct=consts[0], loss_constant=consts[1], value_min=consts[2])
        search_kw = dict(cpuct=consts[0], virtual_loss_const=consts[1], value_min=consts[2], path_cap=consts[3])
    out = mcts_batch.BatchedMCTS(gpu_net, size, num_sim=num_sim, **search_kw).run(cu(roots), seeds=list(range(n)))
    env = ScalarCubeEnv(size)
    for i in range(n):
        env.sim_cube = roots[i].astype(np.int64)
        env.cube = env._observe(env.sim_cube)
        with torch.no_grad():
            acts, used, tree = mcts_ref.solve(cpu_net.predict, env, env.cube, num_sim, random.Random(i), **kw)
        k = int(out["n_actions"][i])
        assert out["actions"][i, :k].tolist() == (acts or []), i
        assert int(out["n_sims"][i]) == used and int(out["n_nodes"][i]) == len(tree.nodes), i
        root = tree.nodes[tree.key(env.cube)]
        assert out["root_N"][i].tolist() == [int(v) for v in root[3]], i
        assert out["root_W"][i].tolist() == [float(v) for v in root[2]], i
        assert out["root_L"][i].tolist() == [int(v) for v in root[4]], i


def test_new_entry_points_edge_cases():
    """Empty and degenerate inputs of the entry points added in round 1."""
    from rubiks_cube_solver_b200 import mcts_batch
    from oracle.gen_golden import ExactSearchNet
    d = dev()
    for size in SIZES:
        a = T.N_ACTIONS[size]
        assert ops.moves_from_seeds(size, [], 10).shape == (0, 10)
        assert ops.moves_from_seeds(size, [3, 4], 0).shape == (2, 0)
        with pytest.raises(ValueError):
            ops.moves_from_seeds(size, [1], 129)
        tv, tp, err = ops.adi_targets(size, torch.empty((0, a), device=d), torch.empty((0, a), dtype=torch.uint8, device=d),
                                      torch.empty(0, device=d), torch.empty(0, dtype=torch.int32, device=d), 1.0)
        assert tv.numel() == 0 and tp.numel() == 0 and err.numel() == 0
        # one tree, already one move from solved: the very first simulation returns [the solving move]
        net = ExactSearchNet(T.STATE_DIM[size], a).to(d)
        root = O.scramble(size, np.array([[2]]))
        out = mcts_batch.BatchedMCTS(net, size, num_sim=5).run(cu(root), seeds=[0])
        assert out["solved"].tolist() == [True] and out["n_sims"].tolist() == [1]
        assert out["actions"][0, :1].tolist() == [3] and int(out["n_actions"][0]) == 1
        with pytest.raises(ValueError):
            mcts_batch.BatchedMCTS(net, size, num_sim=300)
    # the C ABI rejects bad arguments without touching the device
    lib = _lib.load()
    assert lib.cube_moves_from_seeds(3, None, 5, 10, None, None, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_moves_from_seeds(4, None, 0, 10, None, None, None) == _lib.CUBE_ERR_SIZE
    assert lib.cube_adi_targets(3, None, None, None, None, None, 0, 7, None, None, None, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_mcts_traverse(3, None, ctypes.c_float(1.0), 150, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_set_reserved_sms(-1) == _lib.CUBE_ERR_ARG and lib.cube_set_reserved_sms(0) == 0


def test_peer_allreduce_single_rank_and_argument_checks():
    """C ABI cube_peer_allreduce_i64 with a world of one (the exchange buffer is plain device memory): the sum of
    one rank's values is the values, call after call (epochs 1, 2, 3: both slot parities), and the argument checks."""
    lib = _lib.load()
    dev = torch.device("cuda", 0)
    cap = 64
    nbytes = lib.cube_peer_buffer_bytes(cap)
    assert nbytes > 0 and nbytes % 128 == 0 and lib.cube_peer_buffer_bytes(0) == _lib.CUBE_ERR_ARG
    buf = torch.zeros(nbytes // 8, dtype=torch.int64, device=dev)
    ptrs = (ctypes.c_uint64 * 1)(buf.data_ptr())
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    for epoch in (1, 2, 3):
        v = torch.arange(-5, cap - 5, dtype=torch.int64, device=dev) * (2 ** 33 + epoch)
        want = v.clone()
        assert lib.cube_peer_allreduce_i64(1, 0, ptrs, ctypes.c_void_p(v.data_ptr()), cap, cap, epoch, stream) == 0
        assert torch.equal(v, want)
    v = torch.ones(8, dtype=torch.int64, device=dev)
    p = ctypes.c_void_p(v.data_ptr())
    E = _lib.CUBE_ERR_ARG
    assert lib.cube_peer_allreduce_i64(0, 0, ptrs, p, 8, cap, 4, stream) == E          # world
    assert lib.cube_peer_allreduce_i64(9, 0, ptrs, p, 8, cap, 4, stream) == E
    assert lib.cube_peer_allreduce_i64(1, 1, ptrs, p, 8, cap, 4, stream) == E          # rank
    assert lib.cube_peer_allreduce_i64(1, 0, ptrs, p, cap + 1, cap, 4, stream) == E    # n > capacity
    assert lib.cube_peer_allreduce_i64(1, 0, ptrs, p, 8, cap, 0, stream) == E          # epoch 0
    assert lib.cube_peer_allreduce_i64(1, 0, None, p, 8, cap, 4, stream) == E
    odd = (ctypes.c_uint64 * 1)(buf.data_ptr() + 8)
    assert lib.cube_peer_allreduce_i64(1, 0, odd, p, 8, cap, 4, stream) == _lib.CUBE_ERR_ALIGN
    assert lib.cube_peer_allreduce_i64(1, 0, ptrs, p, 0, cap, 4, stream) == 0          # nothing to do
    torch.cuda.synchronize()


def test_peer_allreduce_two_ranks():
    """The peer-memory all-reduce against torch.distributed's on two GPUs (tools/peer_allreduce_check.py under
    torchrun: 200 calls with rank-dependent delays + three unsynchronised calls in a row)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29533",
                          os.path.join(root, "tools", "peer_allreduce_check.py")],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["world"] == 2 and line["mismatching_calls"] == 0


def test_two_devices_in_one_process():
    """Launch state (dynamic shared-memory opt-in, scheduler slots, SM count) is kept per device."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    rng = np.random.RandomState(2)
    for size in SIZES:
        a = T.N_ACTIONS[size]
        moves = rng.randint(a, size=(64 * 50 + 7, 30)).astype(np.uint8)
        want = O.scramble(size, moves)
        act = rng.randint(a, size=moves.shape[0]).astype(np.uint8)
        for d in (1, 0, 1):
            device = torch.device("cuda", d)
            st, so, _ = ops.scramble(size, torch.from_numpy(moves).to(device))
            assert st.device == device and (st.cpu().numpy() == want).all()
            stepped, _, _ = ops.step(size, st, torch.from_numpy(act).to(device))
            assert (stepped.cpu().numpy() == O.apply_moves(size, want, act)).all()
            res = ops.expand(size, stepped[:100].contiguous(), dtype=torch.bfloat16, want_children=True)
            assert (res["children"].cpu().numpy() == O.expand(size, O.apply_moves(size, want, act)[:100])[0]).all()


@pytest.mark.parametrize("size", SIZES)
def test_host_cube_single_cube_calls(size):
    """C ABI cube_env_host_* (mapped pinned page, one synchronisation per call): step / scramble / encode
    of one cube against the oracle, the no-move index, depth 0, and the argument checks."""
    rng = np.random.RandomState(size)
    A, S = T.N_ACTIONS[size], T.N_STICKERS[size]
    hc = ops.HostCube(size, max_depth=64)
    moves = rng.randint(A, size=40).astype(np.uint8)
    st, oh, solved = hc.scramble(moves)
    want = O.scramble(size, moves[None, :])[0]
    assert st.dtype == np.uint8 and (st == want).all() and not solved
    assert (oh == O.encode(size, want[None])[0]).all() and (hc.encode(st) == oh).all()
    cur = st
    for a in rng.randint(A, size=30):
        cur, oh, solved = hc.step(cur, int(a))
        want = O.scramble(size, np.array([[a]]), init=want[None])[0]
        assert (cur == want).all() and (oh == O.encode(size, want[None])[0]).all()
        assert solved == bool(O.is_solved(size, want[None])[0])
    back = np.concatenate([moves[:6], moves[:6][::-1] ^ 1]).astype(np.uint8)
    st, oh, solved = hc.scramble(back)
    assert solved and (st == O.scramble(size, np.zeros((1, 0), dtype=np.uint8))[0]).all()
    st0, _, solved0 = hc.scramble(np.zeros(0, dtype=np.uint8))                 # depth 0: the solved cube
    assert solved0 and (st0 == st).all()
    same, _, _ = hc.step(cur, 12)                                              # CUBE_NOOP
    assert (same == cur).all()
    with pytest.raises(ValueError):
        hc.scramble(np.zeros(65, dtype=np.uint8))
    hc.close()


@pytest.mark.parametrize("size,depth", [(3, 30), (3, 32), (3, 24), (3, 128), (2, 20), (2, 32), (2, 33), (2, 96)])
def test_scramble_many_tiles_per_warp(size, depth):
    """Two persistent CTAs (cube_set_reserved_sms): every warp walks many tiles, so both move buffers, the
    barriers' phase bits, the out-tile hand-over to the bulk store and the dynamic tail are exercised far
    beyond what a full-width launch of a test-sized batch reaches."""
    rng = np.random.RandomState(7 * depth + size)
    n = 64 * 900 + 17
    moves = rng.randint(T.N_ACTIONS[size], size=(n, depth)).astype(np.uint8)
    ops.set_reserved_sms(ops.sm_count() - 2)
    try:
        states, solved, reward = ops.scramble(size, cu(moves))
        torch.cuda.synchronize()
    finally:
        ops.set_reserved_sms(0)
    want, ws, wr, _ = C.scramble(size, moves)
    assert (states.cpu().numpy() == want).all()
    assert (solved.cpu().numpy().astype(bool) == ws).all() and (reward.cpu().numpy() == wr).all()


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("n", (1, 15, 16, 17, 1000))
def test_expand_codes_equal_argmax_of_the_onehot_rows(size, n):
    """cube_expand_codes: compact codes = argmax over every one-hot row of cube_expand's output, zero-padded;
    children, verdicts and the parent's one-hot identical to cube_expand's."""
    rng = np.random.RandomState(n + size)
    A = T.N_ACTIONS[size]
    states = cu(O.scramble(size, rng.randint(A, size=(n, 9))))
    states[0] = cu(O.scramble(size, np.zeros((1, 0), dtype=np.int64)))[0]          # solved parent: its children are one move away
    want = ops.expand(size, states, dtype=torch.uint8, want_children=True, want_parent_onehot=True)
    got = ops.expand_codes(size, states, parent_dtype=torch.float32, want_children=True)
    r, key = T.STATE_DIM[size][0], ops.key_bytes(size)
    assert got["child_codes"].shape == (n, A, key) and got["parent_codes"].shape == (n, key)
    assert (got["child_codes"][..., :r] == want["child_onehot"].argmax(-1).to(torch.uint8)).all()
    assert (got["parent_codes"][..., :r] == want["parent_onehot"].argmax(-1).to(torch.uint8)).all()
    assert (got["child_codes"][..., r:] == 0).all() and (got["parent_codes"][..., r:] == 0).all()
    assert (got["children"] == want["children"]).all() and (got["solved"] == want["solved"]).all()
    assert (got["reward"] == want["reward"]).all()
    assert (got["parent_onehot"] == want["parent_onehot"].float()).all()


# ------------------------------------------------------------------ round 2: paths that had no test
def _guarded(n_bytes, dtype=torch.uint8, guard=4096, fill=0xA5):
    """A device buffer with `guard` canary bytes on both sides of the n_bytes payload (16-byte aligned)."""
    raw = torch.full((guard + n_bytes + 15 + guard,), fill, dtype=torch.uint8, device=dev())
    pad = (-(raw.data_ptr() + guard)) % 16
    lo = guard + pad
    view = raw[lo:lo + n_bytes].view(dtype)
    return raw, view, lo


def _guards_intact(raw, lo, n_bytes, fill=0xA5):
    return bool((raw[:lo] == fill).all()) and bool((raw[lo + n_bytes:] == fill).all())


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("depth", (1, 7, 20, 30, 32, 64, 97, 200, 321, 400))
def test_garbage_action_bytes_are_memory_safe_scramble(size, depth):
    """include/cube_b200.h: action bytes 13..255 are memory-safe but give unspecified states.  Rows whose
    moves are all valid must still be exact, the guard bytes around every output must survive, and the
    device must not fault -- on every scramble variant (flat / swizzled / four-per-lane K1p at depth
    <= 320, the ragged tile kernel, the deep kernel)."""
    rng = np.random.RandomState(1000 * size + depth)
    S, A = T.N_STICKERS[size], T.N_ACTIONS[size]
    n = 64 * 148 * 3 + 37                                              # whole K1p tiles + a ragged tail
    moves = rng.randint(A, size=(n, depth)).astype(np.uint8)
    bad_rows = rng.choice(n, n // 3, replace=False)
    for r in bad_rows[: len(bad_rows) // 2]:                            # one garbage byte somewhere
        moves[r, rng.randint(depth)] = rng.randint(13, 256)
    for r in bad_rows[len(bad_rows) // 2:]:                             # all garbage
        moves[r] = rng.randint(13, 256, size=depth)
    moves[bad_rows[0]] = 255
    good = np.ones(n, dtype=bool)
    good[bad_rows] = False
    raw_s, states, lo_s = _guarded(n * S)
    raw_f, solved, lo_f = _guarded(n)
    raw_r, reward, lo_r = _guarded(4 * n, torch.float32)
    counters = ops.new_counters(dev())
    ops.scramble(size, cu(moves), out=states.view(n, S), solved=solved, reward=reward, counters=counters)
    torch.cuda.synchronize()                                           # a fault would surface here
    assert _guards_intact(raw_s, lo_s, n * S) and _guards_intact(raw_f, lo_f, n) and _guards_intact(raw_r, lo_r, 4 * n)
    want, ws, wr, _ = C.scramble(size, moves[good])
    assert (states.view(n, S).cpu().numpy()[good] == want).all()
    assert (solved.cpu().numpy()[good].astype(bool) == ws).all() and (reward.cpu().numpy()[good] == wr).all()
    assert set(np.unique(solved.cpu().numpy())) <= {0, 1} and set(np.unique(reward.cpu().numpy())) <= {-1.0, 1.0}
    assert int(counters[1]) == n
    with pytest.raises(IndexError):
        ops.validate_actions(size, cu(moves))


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("depth", (1, 5, 64, 65))
def test_garbage_action_bytes_are_memory_safe_step_and_walk(size, depth):
    """The same canary for cube_step / cube_walk (K2p at depth <= 64, the tile kernel beyond and for the tail)."""
    rng = np.random.RandomState(77 * size + depth)
    S, A = T.N_STICKERS[size], T.N_ACTIONS[size]
    n = 64 * 148 * 2 + 29
    start = O.scramble(size, rng.randint(A, size=(n, 9)))
    moves = rng.randint(A, size=(n, depth)).astype(np.uint8)
    bad_rows = rng.choice(n, n // 4, replace=False)
    for r in bad_rows:
        moves[r, rng.randint(depth)] = rng.randint(13, 256)
    moves[bad_rows[0]] = 255
    good = np.ones(n, dtype=bool)
    good[bad_rows] = False
    raw_s, out, lo_s = _guarded(n * S)
    raw_f, solved, lo_f = _guarded(n)
    raw_r, reward, lo_r = _guarded(4 * n, torch.float32)
    ops.walk(size, cu(start), cu(moves), out=out.view(n, S), solved=solved, reward=reward)
    torch.cuda.synchronize()
    assert _guards_intact(raw_s, lo_s, n * S) and _guards_intact(raw_f, lo_f, n) and _guards_intact(raw_r, lo_r, 4 * n)
    want = O.scramble(size, moves[good], init=start[good])
    assert (out.view(n, S).cpu().numpy()[good] == want).all()
    assert (solved.cpu().numpy()[good].astype(bool) == O.is_solved(size, want)).all()
    if depth == 1:                                                      # cube_step, in place
        raw_i, st, lo_i = _guarded(n * S)
        st.view(n, S).copy_(cu(start))
        ops.step(size, st.view(n, S), cu(moves[:, 0]), solved=solved, reward=reward)
        torch.cuda.synchronize()
        assert _guards_intact(raw_i, lo_i, n * S)
        assert (st.view(n, S).cpu().numpy()[good] == want).all()


@pytest.mark.parametrize("size", SIZES)
def test_sliced_and_offset_buffers(size):
    """ADVICE r1: `ops.step(size, states, actions_all[t])` on a [T, N] tensor with N % 16 != 0, or a sliced
    solved= / reward= buffer, is contiguous but not 16- / 8- / 4-byte aligned.  Such calls must work (the byte-wise
    kernels take them), not fault."""
    rng = np.random.RandomState(size)
    S, A = T.N_STICKERS[size], T.N_ACTIONS[size]
    n, steps = 64 * 300 + 13, 3                                        # N % 16 == 13
    start = O.scramble(size, rng.randint(A, size=(n, 8)))
    actions_all = cu(rng.randint(A, size=(steps, n)).astype(np.uint8))
    flags = torch.zeros(steps * n + 3, dtype=torch.uint8, device=dev())
    rewards = torch.zeros(steps * n + 3, dtype=torch.float32, device=dev())
    states, want = cu(start), start
    for t in range(steps):
        so = flags[1 + t * n:1 + (t + 1) * n]                          # odd byte offset
        rw = rewards[1 + t * n:1 + (t + 1) * n]                        # 4-byte but not 8-byte aligned
        ops.step(size, states, actions_all[t], solved=so, reward=rw)
        want = O.apply_moves(size, want, actions_all[t].cpu().numpy())
        assert (states.cpu().numpy() == want).all()
        assert (so.cpu().numpy().astype(bool) == O.is_solved(size, want)).all()
        assert (rw.cpu().numpy() == O.rewards(O.is_solved(size, want))).all()
    moves = rng.randint(A, size=(n, 30)).astype(np.uint8)
    so, rw = flags[1:1 + n], rewards[1:1 + n]
    st, _, _ = ops.scramble(size, cu(moves), solved=so, reward=rw)
    w2, ws, wr, _ = C.scramble(size, moves)
    assert (st.cpu().numpy() == w2).all() and (so.cpu().numpy().astype(bool) == ws).all() and (rw.cpu().numpy() == wr).all()
    # walk with a move array that starts 1 byte into an allocation
    mv = torch.zeros(n * 4 + 1, dtype=torch.uint8, device=dev())
    mv[1:] = cu(moves[:, :4]).reshape(-1)
    out, so2, _ = ops.walk(size, cu(start), mv[1:].view(n, 4))
    assert (out.cpu().numpy() == O.scramble(size, moves[:, :4], init=start)).all()


@pytest.mark.parametrize("size", SIZES)
def test_reset_without_seed_draws_from_and_rewinds_the_global_rng(size):
    """reset(seed=None) (cube_env.py:60-68): the moves come from the GLOBAL legacy generator and the
    generator is put back, so two resets in a row give the same cube and the stream is not advanced --
    against oracle/scalar_env.py (pinned to the reference by tests/test_oracle_vs_reference.py)."""
    from oracle.scalar_env import ScalarCubeEnv
    env, ref = R.make_env(torch.device("cpu"), size), ScalarCubeEnv(size)
    for seed0, k in ((5, 1), (123, 7), (2 ** 31 + 7, 30)):
        np.random.seed(seed0)
        before = np.random.get_state()
        obs = env.reset(scramble_count=k)
        mid = np.random.get_state()
        want_obs = ref.reset(scramble_count=k)
        assert (np.random.get_state()[1] == before[1]).all() and np.random.get_state()[2] == before[2]
        assert (mid[1] == before[1]).all() and mid[2] == before[2]                  # rewound by the drop-in too
        assert (env.sim_cube == ref.sim_cube).all() and (obs == want_obs).all() and obs.dtype == want_obs.dtype
        assert (env.sim_cube == O.scramble(size, np.random.RandomState(seed0).randint(T.N_ACTIONS[size], size=k)[None])[0]).all()
        again = env.reset(seed=None, scramble_count=k)                              # same stream position -> same cube
        assert (again == obs).all()
        np.random.randint(10)                                                       # advance the stream: another cube
        other = env.reset(scramble_count=k)
        ref.reset(scramble_count=k)
        assert (env.sim_cube == ref.sim_cube).all() and (other == ref.cube).all()
    with pytest.raises(UnboundLocalError):
        env.reset(scramble_count=0)


def test_config3_whole_on_one_gpu_64Mi():
    """SURVEY.md section 8d config 3 as ONE device's job: 64 Mi instances x depth 30 (2 GB of moves, 3.6 GB of
    sticker rows) -- 32-bit tile indices, > 2^31 byte offsets and the dynamic-tail scheduler at 1 Mi tiles."""
    size, n, depth = 3, 64 * 2 ** 20, 30
    gen = torch.Generator(device=dev()).manual_seed(1234)
    moves = torch.randint(0, 12, (n, depth), dtype=torch.uint8, device=dev(), generator=gen)
    back = torch.randint(0, n, (1000,), device=dev(), generator=gen)
    moves[back, 15:] = moves[back, :15].flip(1) ^ 1                                # rows that come back to solved
    counters = ops.new_counters(dev())
    states, solved, reward = ops.scramble(size, moves, counters=counters)
    idx = np.concatenate((np.arange(4096), n - 1 - np.arange(4096), np.random.RandomState(7).randint(n, size=8192),
                          back.cpu().numpy()))
    want, ws, wr, _ = C.scramble(size, moves[idx].cpu().numpy())
    assert (states[idx].cpu().numpy() == want).all()
    assert (solved[idx].cpu().numpy().astype(bool) == ws).all() and (reward[idx].cpu().numpy() == wr).all()
    assert ws[-1000:].all()
    sub = slice(n - 2 ** 20 - 77, n - 77)
    _, _, _, cnt = C.scramble(size, moves[sub].cpu().numpy())
    assert int(solved[sub].sum()) == cnt
    assert int(counters[0]) == int(solved.sum()) >= len(set(back.tolist())) and int(counters[1]) == n
    assert float(reward.double().sum()) == 2 * int(counters[0]) - n
    # checksum of checksums: every row is a permutation of the solved multiset
    ok = torch.ones(n, dtype=torch.bool, device=dev())
    for c in range(6):
        ok &= (states == c).sum(dim=1) == 9
    assert bool(ok.all())
    del ok
    # scramble o inverse = identity for all 64 Mi rows, in two halves (the 60-move array is 4 GB)
    for half in range(2):
        m = moves[half * (n // 2):(half + 1) * (n // 2)]
        undo = torch.cat((m, m.flip(1) ^ 1), dim=1).contiguous()
        counters.zero_()
        s2, so2, _ = ops.scramble(size, undo, counters=counters)
        assert int(counters[0]) == n // 2 and bool(so2.all())
        del undo, s2, so2
    # one step on the resident rows == a depth-31 scramble
    extra = torch.randint(0, 12, (n,), dtype=torch.uint8, device=dev(), generator=gen)
    stepped, so3, _ = ops.step(size, states, extra)
    longer, so4, _ = ops.scramble(size, torch.cat((moves, extra[:, None]), dim=1).contiguous())
    assert bool((stepped == longer).all()) and bool((so3 == so4).all())


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("n", (1, 15, 16, 17, 1000, 70001))
def test_expand_codes_vs_oracle(size, n):
    """cube_expand_codes against the ORACLE (not against cube_expand): codes = the column of the 1 of every
    one-hot row of oracle.cube_np.encode, through the reference's tables as shipped."""
    rng = np.random.RandomState(3 * n + size)
    A, S = T.N_ACTIONS[size], T.N_STICKERS[size]
    r, key = T.STATE_DIM[size][0], ops.key_bytes(size)
    parents = O.scramble(size, rng.randint(A, size=(n, 10)))
    parents[0] = O.scramble(size, np.array([[5]]))[0]
    got = ops.expand_codes(size, cu(parents), parent_dtype=torch.uint8, want_children=True)
    want_c, want_s = O.expand(size, parents)
    assert (got["children"].cpu().numpy() == want_c).all()
    assert (got["solved"].cpu().numpy().astype(bool) == want_s).all() and got["solved"][0, 4] == 1
    assert (got["reward"].cpu().numpy() == np.where(want_s, 1.0, -1.0)).all()
    enc_c = O.encode(size, want_c.reshape(n * A, S)).reshape(n, A, r, -1)
    enc_p = O.encode(size, parents)
    assert (enc_c.sum(-1) == 1).all() and (enc_p.sum(-1) == 1).all()
    assert (got["child_codes"].cpu().numpy()[..., :r] == enc_c.argmax(-1)).all()
    assert (got["parent_codes"].cpu().numpy()[..., :r] == enc_p.argmax(-1)).all()
    assert (got["child_codes"].cpu().numpy()[..., r:] == 0).all() and (got["parent_codes"].cpu().numpy()[..., r:] == 0).all()
    assert (got["parent_onehot"].cpu().numpy() == enc_p).all()


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("n,depth", [(1, 1), (31, 2), (32, 30), (33, 30), (1000, 7), (148 * 8 * 32 * 2 + 5, 30), (4099, 31),
                                     (100, 131), (70, 289), (40, 526), (24, 527), (9, 1160)])
def test_scramble_prefixes_vs_oracle(size, n, depth):
    """cube_scramble_prefixes: every prefix of every scramble in one launch, cube-major
    (get_random_samples' order, cube_env.py:187-194), with the done flag of every prefix -- against the
    oracle's per-step states.  Depths beyond the single-launch limit go through adi.scramble_prefixes'
    per-level path."""
    rng = np.random.RandomState(n + depth + size)
    A, S = T.N_ACTIONS[size], T.N_STICKERS[size]
    moves = rng.randint(A, size=(n, depth)).astype(np.uint8)
    if depth >= 4:
        moves[::3, 2:4] = moves[::3, :2][:, ::-1] ^ 1                   # solved again after four moves
    _, want, want_solved = O.scramble(size, moves, per_step=True)
    if depth <= ops.prefixes_max_depth(size):
        counters = ops.new_counters(dev())
        got, solved = ops.scramble_prefixes(size, cu(moves), want_solved=True, counters=counters)
        assert got.shape == (n, depth, S) and (got.cpu().numpy() == want).all()
        assert (solved.cpu().numpy().astype(bool) == want_solved).all()
        assert counters.tolist()[:2] == [int(want_solved.sum()), n * depth]
        if depth >= 4:
            assert solved[0, 3] == 1
    else:
        with pytest.raises(ValueError):
            ops.scramble_prefixes(size, cu(moves))
    assert (adi.scramble_prefixes(size, cu(moves)).cpu().numpy() == want).all()
    assert ops.prefixes_max_depth(size) == (526 if size == 3 else 1159)


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("obs_dtype", (torch.float32, torch.bfloat16))
def test_batched_mcts_graph_replay_equals_eager_and_golden(size, obs_dtype):
    """BatchedMCTS(graph=True) replays simulations 2.. as one captured CUDA graph (the simulation index lives on
    the device): same searches as the eager loop and as the reference's own mcts.py (golden vectors).  The exact
    net's outputs are exact in bf16 too (one-hot inputs, weights that are multiples of 1/8)."""
    from rubiks_cube_solver_b200 import mcts_batch
    from oracle.gen_golden import ExactSearchNet, MCTS_CFG
    g = golden("mcts_%d.npz" % size)
    cases = g["cases"]
    roots = np.stack([O.scramble(size, O.reference_moves(size, int(sd), int(d))[None])[0] for sd, d in cases])
    net = ExactSearchNet(T.STATE_DIM[size], T.N_ACTIONS[size]).to(dev())
    cfg = MCTS_CFG["mcts"]
    outs = []
    for graph in (False, True):
        search = mcts_batch.BatchedMCTS(net, size, num_sim=cfg["numMCTSSim"], cpuct=cfg["cpuct"], obs_dtype=obs_dtype,
                                        virtual_loss_const=cfg["virtual_loss_const"], value_min=cfg["value_min"], graph=graph)
        outs.append(search.run(cu(roots), seeds=[1000 + int(sd) for sd, _ in cases]))
    for out in outs:
        assert (out["n_sims"].cpu().numpy() == g["n_sims"]).all() and (out["n_actions"].cpu().numpy() == g["n_actions"]).all()
        assert (out["actions"].cpu().numpy()[:, :g["actions"].shape[1]] == g["actions"]).all()
        assert (out["n_nodes"].cpu().numpy() == g["n_nodes"]).all()
        assert (out["root_N"].cpu().numpy() == g["root_N"]).all() and (out["root_L"].cpu().numpy() == g["root_L"]).all()
        assert (out["root_W"].cpu().numpy().astype(np.float64) == g["root_W"]).all()


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("num_sim", (1, 2, 3, 4, 30, 50))
def test_batched_mcts_short_searches_full_action_lists(size, num_sim):
    """ADVICE r1: a traversal may bounce (U then U' is back at the root's key), so a returned path can be longer
    than num_sim + 1; the action list must come back whole (n_actions <= actions.shape[1]) and equal to the
    per-cube search of oracle/mcts_ref.py.  Many shallow cubes, tiny simulation budgets."""
    import random
    from rubiks_cube_solver_b200 import mcts_batch
    from oracle import mcts_ref
    from oracle.gen_golden import ExactSearchNet
    from oracle.scalar_env import ScalarCubeEnv
    n = 300 if num_sim < 30 else 60
    rng = np.random.RandomState(31 * num_sim + size)
    A = T.N_ACTIONS[size]
    depths = rng.randint(1, 5 if num_sim < 50 else 9, size=n)      # deeper roots: longer searches, more transpositions
    roots = np.stack([O.scramble(size, rng.randint(A, size=(1, int(d))))[0] for d in depths])
    gpu_net = ExactSearchNet(T.STATE_DIM[size], A).to(dev())
    cpu_net = ExactSearchNet(T.STATE_DIM[size], A)
    out = mcts_batch.BatchedMCTS(gpu_net, size, num_sim=num_sim, graph=(num_sim == 30)).run(cu(roots), seeds=list(range(n)))
    assert num_sim < 50 or not bool(out["solved"].all())             # some trees run their whole budget
    assert int(out["n_actions"].max()) <= out["actions"].shape[1]
    env = ScalarCubeEnv(size)
    for i in range(n):
        env.sim_cube = roots[i].astype(np.int64)
        env.cube = env._observe(env.sim_cube)
        with torch.no_grad():
            acts, used, tree = mcts_ref.solve(cpu_net.predict, env, env.cube, num_sim, random.Random(i))
        k = int(out["n_actions"][i])
        assert out["actions"][i, :k].tolist() == (acts or []), i
        assert (out["actions"][i, k:] == -1).all()
        assert int(out["n_sims"][i]) == used and int(out["n_nodes"][i]) == len(tree.nodes), i
        if acts:                                                         # the returned list solves the cube
            s = roots[i][None]
            for a in acts:
                s = O.apply_moves(size, s, np.array([a]))
            assert O.is_solved(size, s)[0]


def test_batched_mcts_rejects_bad_random_actions():
    from rubiks_cube_solver_b200 import mcts_batch
    from oracle.gen_golden import ExactSearchNet
    net = ExactSearchNet(T.STATE_DIM[2], 6).to(dev())
    roots = cu(O.scramble(2, np.array([[0, 2, 4]])))
    table = torch.full((1, 64), 6, dtype=torch.uint8)
    with pytest.raises(IndexError):
        mcts_batch.BatchedMCTS(net, 2, num_sim=4).run(roots, rand_table=table)


def test_host_reset_pipeline_from_seeds_and_hugepage_buffers():
    """cube_pipeline_reset_host: batched reset(seed, k) for host arrays (4 bytes per cube on the way in, moves
    drawn on the device) against np.random.RandomState(seed).randint + the oracle; outputs land in huge-page
    buffers from cube_host_alloc; solved / reward arrays are optional."""
    for size, depth in ((3, 30), (2, 10)):
        n = 200000 + 77
        seeds = torch.arange(n, dtype=torch.int64) * 7 + 3
        seeds[5] = 2 ** 32 - 1
        packed = torch.where(seeds >= 2 ** 31, seeds - 2 ** 32, seeds).to(torch.int32).contiguous()
        pipe = ops.HostScramblePipeline(size, depth, chunk_instances=1 << 16, n_stages=3)
        states_buf = ops.host_buffer((n, T.N_STICKERS[size]))
        states, solved, reward, count = pipe.reset(packed, states_out=states_buf)
        assert states.data_ptr() == states_buf.data_ptr() and states.data_ptr() % (2 << 20) == 0
        moves = np.stack([np.random.RandomState(int(s)).randint(T.N_ACTIONS[size], size=depth) for s in seeds[:3000]])
        want, ws, wr, _ = C.scramble(size, moves.astype(np.uint8))
        assert (states[:3000].numpy() == want).all() and (solved[:3000].numpy().astype(bool) == ws).all()
        assert (reward[:3000].numpy() == wr).all()
        dev_moves = ops.moves_from_seeds(size, seeds, depth)
        dev_states, dev_solved, _ = ops.scramble(size, dev_moves)
        assert (states.numpy() == dev_states.cpu().numpy()).all() and count == int(dev_solved.sum())
        s2, so2, rw2, c2 = pipe.reset(packed[:1000].contiguous(), want_solved=False, want_reward=False)
        assert so2 is None and rw2 is None and (s2.numpy() == want[:1000]).all() and c2 == int(ws[:1000].sum())
        s3, so3, rw3, _ = pipe.run(torch.from_numpy(moves.astype(np.uint8)), want_reward=False)
        assert rw3 is None and (s3.numpy() == want).all() and (so3.numpy().astype(bool) == ws).all()
        pipe.close()
        with pytest.raises(ValueError):
            ops.HostScramblePipeline(size, 129, chunk_instances=1 << 12).reset(packed[:10].contiguous())
    ops.release_host_buffers()


def test_exact_3x3_encoding_roundtrip_and_reference_mode_unchanged():
    """SURVEY.md section 8f4: the opt-in exact 3x3x3 encoding (encoding="exact": un-mirrored corner slot 6, every
    corner rotation assigned) is a bijection -- decode(encode(s)) == s on a million random states, in every
    dtype -- and equals the NumPy spec (oracle.cube_np.encode_exact); the default stays the reference's lossy
    table bit for bit (py333.py:140-180) and stays un-decodable (cube_env.py:171-172)."""
    n = 10 ** 6
    gen = torch.Generator(device=dev()).manual_seed(8)
    states, _, _ = ops.scramble(3, torch.randint(0, 12, (n, 40), dtype=torch.uint8, device=dev(), generator=gen),
                                want_flags=False)
    states[0] = ops.solved_states(3, 1, dev())[0]
    sample = states[:50000].cpu().numpy()
    for dt in (torch.uint8, torch.bfloat16, torch.float32):
        enc = ops.encode(3, states, dtype=dt, encoding="exact")
        assert bool((ops.decode(3, enc, encoding="exact") == states).all()), dt
        got, clean = onehot_to_u8(enc[:50000])
        assert clean and (got == O.encode_exact(sample)).all(), dt
        del enc
    # one 1 per row; pieces form a permutation; twists sum to 0 mod 3, flips to 0 mod 2
    cols = ops.encode(3, states, dtype=torch.uint8, encoding="exact").argmax(-1)
    assert bool((cols[:, :8].div(3, rounding_mode="floor").sort(dim=1).values == torch.arange(8, device=dev())).all())
    assert bool((cols[:, 8:].div(2, rounding_mode="floor").sort(dim=1).values == torch.arange(12, device=dev())).all())
    assert bool(((cols[:, :8] % 3).sum(1) % 3 == 0).all()) and bool(((cols[:, 8:] % 2).sum(1) % 2 == 0).all())
    # the reference mode is what it was: the shipped table, different from the exact one, not decodable
    ref, _ = onehot_to_u8(ops.encode(3, states[:50000].contiguous(), dtype=torch.uint8))
    assert (ref == O.encode(3, sample)).all() and not (ref == O.encode_exact(sample)).all()
    assert (ref[:, 8:] == O.encode_exact(sample)[:, 8:]).all()                    # edges are the same in both
    with pytest.raises(NotImplementedError):
        ops.decode(3, ops.encode(3, states[:16].contiguous(), dtype=torch.uint8))
    with pytest.raises(ValueError):
        ops.encode(3, states[:16].contiguous(), encoding="lossless")
    # expansion in the exact encoding: children's one-hot rows and compact codes
    par = states[:4099].contiguous()
    res = ops.expand(3, par, dtype=torch.bfloat16, want_children=True, want_parent_onehot=True, encoding="exact")
    wc, ws = O.expand(3, par.cpu().numpy())
    assert (res["children"].cpu().numpy() == wc).all() and (res["solved"].cpu().numpy().astype(bool) == ws).all()
    got, clean = onehot_to_u8(res["child_onehot"])
    assert clean and (got.reshape(-1, 20, 24) == O.encode_exact(wc.reshape(-1, 54))).all()
    assert bool((ops.decode(3, res["child_onehot"].view(-1, 20, 24), encoding="exact").view(-1, 12, 54) == res["children"]).all())
    codes = ops.expand_codes(3, par, encoding="exact")
    assert (codes["child_codes"].cpu().numpy() == O.onehot_columns_exact(wc.reshape(-1, 54)).reshape(-1, 12, 20)).all()
    assert (codes["parent_codes"].cpu().numpy() == O.onehot_columns_exact(par.cpu().numpy())).all()
    # 2x2x2 has one encoding: both names give py222's
    s2, _, _ = ops.scramble(2, torch.randint(0, 6, (5000, 14), dtype=torch.uint8, device=dev(), generator=gen), want_flags=False)
    assert bool((ops.encode(2, s2, dtype=torch.uint8, encoding="exact") == ops.encode(2, s2, dtype=torch.uint8)).all())
    assert bool((ops.decode(2, ops.encode(2, s2, dtype=torch.uint8), encoding="exact") == s2).all())
    # ragged sizes of the decode kernels, every dtype
    for m in (1, 63, 64, 65, 1000):
        for dt in (torch.uint8, torch.bfloat16, torch.float32):
            e = ops.encode(3, states[:m].contiguous(), dtype=dt, encoding="exact")
            assert bool((ops.decode(3, e, encoding="exact") == states[:m]).all())
            e2 = ops.encode(2, s2[:m].contiguous(), dtype=dt)
            assert bool((ops.decode(2, e2) == s2[:m]).all())
            assert (ops.decode(2, e2).cpu().numpy() == O.decode_2(onehot_to_u8(e2)[0])).all()


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("n,depth", [(1, 1), (63, 30), (64 * 148 * 3 + 37, 30), (5000, 20), (4099, 31), (3000, 32), (777, 0),
                                     (2000, 200), (1500, 321), (130, 400)])
def test_scramble_step_fused_equals_scramble_then_step(size, n, depth):
    """cube_scramble_step: `reset` then `step(a)` in one launch (configs[2] read literally) == the oracle's
    scramble of [moves | action] == cube_scramble followed by cube_step, on every scramble variant (K1p flat /
    swizzled / four-per-lane, the tile kernel's ragged tail, the deep kernel); rows whose action undoes the
    last move of a 2-move identity come back solved."""
    rng = np.random.RandomState(5 * n + depth + size)
    A = T.N_ACTIONS[size]
    moves = rng.randint(A, size=(n, depth)).astype(np.uint8)
    act = rng.randint(A, size=n).astype(np.uint8)
    if depth >= 2 and depth % 2 == 1:                                   # a sequence that only the action brings home
        h = depth // 2
        k = min(n, 50)
        moves[:k, h:2 * h] = moves[:k, :h][:, ::-1] ^ 1                  # solved after 2h moves, then one more move ...
        act[:k] = moves[:k, -1] ^ 1                                     # ... which the action undoes
    counters = ops.new_counters(dev())
    states, solved, reward = ops.scramble_step(size, cu(moves), cu(act), counters=counters)
    want, ws, wr, cnt = C.scramble(size, np.concatenate((moves, act[:, None]), axis=1))
    assert (states.cpu().numpy() == want).all()
    assert (solved.cpu().numpy().astype(bool) == ws).all() and (reward.cpu().numpy() == wr).all()
    assert counters.tolist()[:2] == [cnt, n]
    if depth >= 2 and depth % 2 == 1:
        assert ws[:min(n, 50)].all()
    two, _, _ = ops.scramble(size, cu(moves))
    stepped, s2, _ = ops.step(size, two, cu(act))
    assert bool((stepped == states).all()) and bool((s2 == solved).all())
    # an action array at an odd address takes the byte-wise kernels
    off = torch.zeros(n + 1, dtype=torch.uint8, device=dev())
    off[1:] = cu(act)
    st2, _, _ = ops.scramble_step(size, cu(moves), off[1:])
    assert bool((st2 == states).all())


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("depth", (321, 480, 481, 723, 1000))
def test_deep_scrambles_sliced_kernel(size, depth):
    """Depth > 320 (test.py:44 scrambles 1 000 deep): K1p's sliced variant -- move bytes staged 240 per row at a
    time from the 16-byte boundary below each piece, state carried in registers -- with several tiles per warp
    (both buffers, barrier phases across tiles), the last whole tile and the ragged tail through the deep kernel,
    rows that come back to solved, twist pile-ups, and the fused trailing action."""
    rng = np.random.RandomState(depth + 13 * size)
    A = T.N_ACTIONS[size]
    n = 64 * 148 * 4 * 2 + 64 + 29
    moves = rng.randint(A, size=(n, depth)).astype(np.uint8)
    h = depth // 2
    back = rng.choice(n, 400, replace=False)
    moves[back, h:2 * h] = moves[back, :h][:, ::-1] ^ 1
    if depth % 2:
        moves[back, -1] = 12
    if size == 3:
        moves[:64] = np.tile(np.array([2, 4], dtype=np.uint8), (64, depth // 2 + 1))[:, :depth]
    counters = ops.new_counters(dev())
    states, solved, reward = ops.scramble(size, cu(moves), counters=counters)
    clean = np.where(moves == 12, 0, moves)
    want, ws, wr, _ = C.scramble(size, clean)
    if depth % 2:
        want[back], ws[back], wr[back], _ = C.scramble(size, moves[back, :-1])
    assert (states.cpu().numpy() == want).all()
    assert (solved.cpu().numpy().astype(bool) == ws).all() and (reward.cpu().numpy() == wr).all()
    assert counters.tolist()[:2] == [int(ws.sum()), n] and ws[back].all()
    act = rng.randint(A, size=n).astype(np.uint8)
    st2, so2, _ = ops.scramble_step(size, cu(moves), cu(act))
    assert (st2.cpu().numpy() == O.apply_moves(size, want, act)).all()
    assert (so2.cpu().numpy().astype(bool) == O.is_solved(size, O.apply_moves(size, want, act))).all()


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("graph", (False, True))
def test_batched_mcts_reuses_its_tree_store_across_runs(size, graph):
    """A BatchedMCTS keeps its device tree store (and, with graph=True, the captured simulation) between runs over
    batches of the same shape: a second and third search with other roots / seeds must equal fresh searches --
    nothing of the previous trees may leak (stale node keys, memos, counters, action lists)."""
    from rubiks_cube_solver_b200 import mcts_batch
    from oracle.gen_golden import ExactSearchNet
    A = T.N_ACTIONS[size]
    net = ExactSearchNet(T.STATE_DIM[size], A).to(dev())
    rng = np.random.RandomState(size + 40)
    search = mcts_batch.BatchedMCTS(net, size, num_sim=14, graph=graph)
    for rep in range(3):
        n = 96
        roots = np.stack([O.scramble(size, rng.randint(A, size=(1, int(d))))[0] for d in rng.randint(1, 5, size=n)])
        seeds = [int(x) for x in rng.randint(0, 10 ** 6, size=n)]
        got = search.run(cu(roots), seeds=seeds)
        want = mcts_batch.BatchedMCTS(net, size, num_sim=14).run(cu(roots), seeds=seeds)
        for key in ("solved", "n_actions", "n_sims", "n_nodes", "root_N", "root_W", "root_L"):
            assert bool((got[key] == want[key]).all()), (rep, key)
        w = min(got["actions"].shape[1], want["actions"].shape[1])
        assert bool((got["actions"][:, :w] == want["actions"][:, :w]).all())
    search.release()


@pytest.mark.parametrize("size", SIZES)
def test_adi_generate_samples_bf16_passthrough_within_tolerance(size):
    """The ADI iteration with the net in bfloat16: K3's bf16 one-hot buffer reaches the model AS IT IS (no .float()
    pass: the recorded input dtype is bfloat16), chunk by chunk, and the targets agree with the float32 net's within
    bf16 tolerance -- |dV| <= 3e-2 * max(1, |V|) (8-bit mantissa through four layers) -- while everything that is
    integer work (parents' one-hot rows, stickers, solved children, scramble counts) is identical.  The target
    policy may differ only where the float32 values of the best two children are closer than that tolerance."""
    A, (r, c) = T.N_ACTIONS[size], T.STATE_DIM[size]
    nn = torch.nn

    class Net(nn.Module):                                   # DeepCube's shape (model.py:7-45), small hidden sizes
        def __init__(self):
            super().__init__()
            self.enc = nn.Sequential(nn.Flatten(), nn.Linear(r * c, 256), nn.ELU(), nn.Linear(256, 64), nn.ELU())
            self.pol = nn.Sequential(nn.Linear(64, 32), nn.ELU(), nn.Linear(32, A))
            self.val = nn.Sequential(nn.Linear(64, 32), nn.ELU(), nn.Linear(32, 1))
            self.seen = set()

        def forward(self, x):
            self.seen.add(x.dtype)
            if x.dim() == 2:
                x = x.unsqueeze(0)
            h = self.enc(x)
            return self.val(h), self.pol(h)

    torch.manual_seed(size)
    net32 = Net().to(dev())
    net16 = Net().to(dev())
    net16.load_state_dict(net32.state_dict())
    net16 = net16.to(torch.bfloat16)
    rng = np.random.RandomState(size)
    moves = cu(rng.randint(A, size=(700, 9)).astype(np.uint8))
    moves[0, :2] = torch.tensor([4, 5], dtype=torch.uint8)                # back at solved after two moves
    a32 = adi.generate_samples(size, moves, net32, 0.5, forward_chunk=1024)
    a16 = adi.generate_samples(size, moves, net16, 0.5, forward_chunk=1024)
    assert net32.seen == {torch.float32} and net16.seen == {torch.bfloat16}
    assert a32["state"].dtype == torch.float32 and a16["state"].dtype == torch.bfloat16
    assert bool((a16["state"].float() == a32["state"]).all()) and bool((a16["stickers"] == a32["stickers"]).all())
    assert bool((a16["child_solved"] == a32["child_solved"]).all()) and bool((a16["scramble_count"] == a32["scramble_count"]).all())
    tol = 3e-2 * torch.clamp(a32["target_value"].abs(), min=1.0)
    assert bool(((a16["target_value"] - a32["target_value"]).abs() <= tol).all())
    top2 = (a32["child_values"] - 1.0).topk(2, dim=1).values
    clear = ((top2[:, 0] - top2[:, 1]) > 2 * tol) | a32["child_solved"].bool().any(dim=1)
    assert bool((a16["target_policy"][clear] == a32["target_policy"][clear]).all()) and int(clear.sum()) > 100
    assert bool(((a16["error"] - a32["error"]).abs() <= 2 * tol.double()).all())
    # the oracle's rules on the float32 run (cube_env.py:239-252)
    tv, tp, err = O.adi_targets(a32["child_values"].cpu().numpy(), a32["child_solved"].cpu().numpy().astype(bool),
                                a32["parent_values"].cpu().numpy(), a32["scramble_count"].cpu().numpy(), 0.5)
    assert (a32["target_value"].cpu().numpy() == tv).all() and (a32["target_policy"].cpu().numpy() == tp).all()
    assert np.allclose(a32["error"].cpu().numpy(), err, rtol=0, atol=1e-12)


_SCRAMBLE_K = ("test_scramble_vs_oracle_depths or test_scramble_tile_and_depth_boundaries or "
               "test_garbage_action_bytes_are_memory_safe_scramble or test_scramble_swizzled_move_tiles")
_DEEP_K = ("test_deep_scrambles_sliced_kernel or ((test_scramble_vs_oracle_depths or test_scramble_tile_and_depth_boundaries "
           "or test_garbage_action_bytes_are_memory_safe_scramble) and (321 or 400))")
_WALK_K = ("test_walk_tile_and_depth_boundaries or test_walk_vs_oracle_any_bytes or "
           "test_garbage_action_bytes_are_memory_safe_step_and_walk")
# test_optional_outputs_gpu.py: every output set on the same paths
_SCRAMBLE_K += (" or test_scramble_every_output_set or test_scramble_output_sets_many_tiles_per_warp or "
                "test_scramble_partial_flags_unaligned or test_scramble_step_abi_output_sets or "
                "test_noop_padded_reference_scrambles_without_flags or test_host_pipeline_flag_combinations")
_DEEP_K += (" or ((test_scramble_every_output_set or test_scramble_partial_flags_unaligned or "
            "test_scramble_step_abi_output_sets) and (321 or 400))")
_WALK_K += " or test_walk_and_step_abi_output_sets"
# every A/B switch with the tests that reach the path it controls
# K3c (leaf_children_kernel) runs with the children's one-hot rows in bf16 / u8
_K3C_K = "test_expand_vs_oracle or test_expand_every_output_set or test_expand_rows_that_name_a_cubelet_twice"
_SWITCH_K = {
    "CUBE_PAIR_SWIZZLE=0": _SCRAMBLE_K, "CUBE_PAIR_FOUR=0": _SCRAMBLE_K, "CUBE_SCRAMBLE_CLASSIC=1": _SCRAMBLE_K,
    "CUBE_TAIL_DIV=1": _SCRAMBLE_K, "CUBE_PAIR_SLICED=0": _DEEP_K, "CUBE_SLICE=240": _DEEP_K, "CUBE_WALK_CLASSIC=1": _WALK_K,
    "CUBE_PDL=0": _SCRAMBLE_K + " or " + _WALK_K, "CUBE_K3C_TILE=32": _K3C_K, "CUBE_K3C_TILE=8": _K3C_K, "CUBE_ENV_SPIN=0": "test_host_cube_single_cube_calls or test_cube_env_drop_in",
    # 148 SMs - 146: two persistent CTAs, many tiles per warp
    "CUBE_RESERVED_SMS=146": "test_persistent_kernels_on_concurrent_streams_and_in_a_graph or test_scramble_tile_and_depth_boundaries",
}


@pytest.mark.parametrize("switch", list(_SWITCH_K))
def test_fallback_paths_under_ab_switches(switch):
    """The library reads its A/B switches (DESIGN.md 7b) once per process, so every fallback path gets its own
    interpreter: the tests that reach the path a switch controls again, with the switch set.  (The default paths
    are what the rest of this file runs; all switches x the whole scramble / step / walk selection were run by hand
    on the final tree, DESIGN.md 7b.)"""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    name, value = switch.split("=")
    env = dict(os.environ, **{name: value})
    k = _SWITCH_K[switch]
    files = [os.path.join(root, "tests", f) for f in ("test_gpu_parity.py", "test_optional_outputs_gpu.py",
                                                      "test_expand_outputs_gpu.py")]
    out = subprocess.run([sys.executable, "-m", "pytest"] + files + ["-m", "gpu", "-x", "-q", "-p", "no:cacheprovider", "-k", k],
                         capture_output=True, text=True, timeout=600, env=env, cwd=root)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    assert " passed" in out.stdout and " failed" not in out.stdout


def test_concurrent_first_use_from_host_threads():
    """Host threads that make the first calls of a process at the same time: per-device kernel attributes,
    scheduler slots and switches are set up concurrently (ctypes releases the GIL, so the launchers' host code
    really overlaps).  Eight threads behind a barrier, each on its own stream, run every launcher in a different
    order; every output equals the oracle."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = r'''
import threading
import numpy as np
import torch
from rubiks_cube_solver_b200 import _lib, ops
from oracle import cube_np as O
from oracle import tables as T

_lib.load()                                        # loads the library; no launcher has run yet
dev = torch.device("cuda", 0)
rng = np.random.RandomState(23)
n, n_par, n_threads = 5000, 4099, 8


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.uint8)).to(dev)


def verdicts(size, st):
    ok = O.is_solved(size, st)
    return st, ok, O.rewards(ok)


want, calls, step_start = {}, [], {}               # want: the oracle's arrays in the order the call returns them
for size in (2, 3):
    A = T.N_ACTIONS[size]
    for depth in (30, 32, 400):                    # K1p, K1p with swizzled move tiles, sliced K1p
        m = rng.randint(A, size=(n, depth)).astype(np.uint8)
        want["scramble%d_%d" % (size, depth)] = verdicts(size, O.scramble(size, m))
        calls.append(("scramble%d_%d" % (size, depth), lambda st, size=size, m=cu(m): ops.scramble(size, m)))
    start = O.scramble(size, rng.randint(A, size=(n, 9)))
    act = rng.randint(A, size=n).astype(np.uint8)
    step_start[size] = start
    want["step%d" % size] = verdicts(size, O.apply_moves(size, start, act))
    calls.append(("step%d" % size, lambda st, size=size, a=cu(act): ops.step(size, st[size], a)))
    wm = rng.randint(A, size=(n, 5)).astype(np.uint8)
    want["walk%d" % size] = verdicts(size, O.scramble(size, wm, init=start))
    calls.append(("walk%d" % size, lambda st, size=size, x=cu(start), m=cu(wm): ops.walk(size, x, m)))
    par = O.scramble(size, rng.randint(A, size=(n_par, 9)))
    ch, ok = O.expand(size, par)
    ch_oh = O.encode(size, ch.reshape(n_par * A, -1)).reshape(n_par, A, *T.STATE_DIM[size])
    want["adi%d" % size] = (ch, ch_oh, O.encode(size, par), ok, O.rewards(ok))
    calls.append(("adi%d" % size, lambda st, size=size, p=cu(par): tuple(
        ops.expand(size, p, want_children=True, want_parent_onehot=True)[k]
        for k in ("children", "child_onehot", "parent_onehot", "solved", "reward"))))
    if size == 2:                                  # the MCTS leaf shape
        want["leaf2"] = (ch, O.encode(2, par), ok, O.rewards(ok))
        calls.append(("leaf2", lambda st, p=cu(par): tuple(
            ops.expand(2, p, want_children=True, want_child_onehot=False, want_parent_onehot=True)[k]
            for k in ("children", "parent_onehot", "solved", "reward"))))
    pm = rng.randint(A, size=(n, 30)).astype(np.uint8)
    _, trail, flags = O.scramble(size, pm, per_step=True)
    want["prefixes%d" % size] = (trail, flags)
    calls.append(("prefixes%d" % size, lambda st, size=size, m=cu(pm): ops.scramble_prefixes(size, m, want_solved=True)))
torch.cuda.synchronize()

barrier = threading.Barrier(n_threads)
results, errors = [None] * n_threads, []


def worker(i):
    try:
        stream = torch.cuda.Stream(dev)
        st = {size: cu(step_start[size]) for size in (2, 3)}   # cube_step works in place: one copy per thread
        torch.cuda.synchronize()
        order = calls[i * len(calls) // n_threads:] + calls[:i * len(calls) // n_threads]
        with torch.cuda.stream(stream):
            barrier.wait()
            results[i] = {name: fn(st) for name, fn in order}
        stream.synchronize()
    except BaseException as e:                     # noqa: BLE001
        errors.append(repr(e))
        barrier.abort()


threads = [threading.Thread(target=worker, args=(i,)) for i in range(n_threads)]
for t in threads:
    t.start()
for t in threads:
    t.join()
assert not errors, errors
for i, res in enumerate(results):
    for name, exp in want.items():
        got = res[name]
        assert len(got) == len(exp), name
        for g, w in zip(got, exp):
            g = g.float().cpu().numpy() if g.dtype == torch.bfloat16 else g.cpu().numpy()
            assert g.shape == w.shape and (g == w.astype(g.dtype)).all(), (i, name)
print("checked", len(results), "threads x", len(want), "calls")
'''
    out = subprocess.run([sys.executable, "-c", script], capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "checked 8 threads x 15 calls" in out.stdout


def test_bench_dump_outputs(tmp_path):
    """bench.py --dump-outputs: the last timed step's outputs (a seeded row sample, float32 / float64) equal the
    oracle on the benchmark's own seeded moves, and the same arguments with another --steps write the same files."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    n, dumps = 70007, []
    for steps in (2, 3):
        d = str(tmp_path / ("steps%d" % steps))
        out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", str(steps),
                              "--warmup", "1", "--instances-per-gpu", str(n), "--e2e-steps", "2", "--skip-cpu",
                              "--skip-other", "--dump-outputs", d], capture_output=True, text=True, timeout=600, cwd=root)
        assert out.returncode == 0, out.stderr[-3000:]
        line = json.loads(out.stdout.strip().splitlines()[-1])
        assert line["steps"] == steps and line["gpu_launches"] == steps
        dumps.append({f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)})
    a, b = dumps
    assert sorted(a) == ["counters", "reward", "rows", "solved", "states"]
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    for k in a:
        assert a[k].dtype in (np.float32, np.float64) and np.array_equal(a[k], b[k]), k
    gen = torch.Generator(device=dev()).manual_seed(1234)
    moves = torch.randint(0, 12, (n, 30), dtype=torch.uint8, device=dev(), generator=gen).cpu().numpy()
    want = O.scramble(3, moves)
    solved = O.is_solved(3, want)
    rows = a["rows"].astype(np.int64)
    assert rows.size == 1 << 16 and (np.diff(rows) > 0).all() and rows[-1] < n
    assert (a["states"] == want[rows]).all() and (a["solved"] == solved[rows]).all()
    assert (a["reward"] == O.rewards(solved[rows])).all()
    assert a["counters"].tolist() == [int(solved.sum()), n]
