"""The exact 2x2x2 distance table on the device (csrc/distance.cu): the BFS build, the lookup and the optimal solve
against the oracle, garbage rows with guard bytes around the outputs, and rollout.optimal_gap with the reference's
trained 2x2x2 checkpoint against its recorded episodes."""
import ctypes
import hashlib
import os

import numpy as np
import pytest
import torch

from oracle import cube_np as O
from oracle import distance_np as D
from oracle import tables as T

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
SHA256 = "de0634732a9d7224ed4525a24b857253201699fc5a8ac438989403c2da486f04"


def dev():
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def table():
    return D.distance_table_2()


def _scrambles(n, seed, max_depth=40):
    """n sticker rows scrambled on the device, depths 0..max_depth (shorter rows padded with the no-op index)."""
    from rubiks_cube_solver_b200 import ops
    rng = np.random.RandomState(seed)
    moves = rng.randint(6, size=(n, max_depth)).astype(np.uint8)
    moves[np.arange(max_depth)[None, :] >= rng.randint(0, max_depth + 1, size=(n, 1))] = 12
    states, _, _ = ops.scramble(2, torch.from_numpy(moves).to(dev()), want_flags=False)
    return states


def _garbage(seed):
    """Random bytes, colours >= 6, two stickers swapped, a twisted corner."""
    rng = np.random.RandomState(seed)
    good = _scrambles(4000, seed + 1).cpu().numpy()
    rnd = rng.randint(0, 256, size=(1000, 24)).astype(np.uint8)
    colour = good[:1000].copy()
    colour[np.arange(1000), rng.randint(24, size=1000)] = rng.randint(6, 256, size=1000)
    swapped = good[1000:2000].copy()
    for row in swapped:
        i, j = rng.choice(24, size=2, replace=False)
        while row[i] == row[j]:
            i, j = rng.choice(24, size=2, replace=False)
        row[i], row[j] = row[j], row[i]
    twisted = good[2000:3000].copy()
    slots = T.PIECE_DEFS_2[rng.randint(7, size=1000)]
    twisted[np.arange(1000)[:, None], slots] = twisted[np.arange(1000)[:, None], np.roll(slots, 1, axis=1)]
    return np.concatenate([rnd, colour, swapped, twisted, good[3000:]])      # the last 1000 rows are reachable


def _guarded(n_bytes, offset=0, guard=4096, fill=0xA5):
    """A device buffer with `guard` canary bytes on both sides of the payload, which starts `offset` bytes past a
    16-byte boundary."""
    raw = torch.full((guard + 16 + n_bytes + guard,), fill, dtype=torch.uint8, device=dev())
    lo = guard + (-(raw.data_ptr() + guard)) % 16 + offset
    return raw, raw[lo:lo + n_bytes], lo


def _guards_intact(raw, lo, n_bytes, fill=0xA5):
    return bool((raw[:lo] == fill).all()) and bool((raw[lo + n_bytes:] == fill).all())


def test_device_table_equals_the_oracle_table(table):
    from rubiks_cube_solver_b200 import _lib, ops
    t = ops.distance_table(dev())
    assert t.dtype == torch.uint8 and t.shape == (3674160,) and ops.distance_table(dev()) is t      # cached
    got = t.cpu().numpy()
    assert (got == table).all() and hashlib.sha256(got.tobytes()).hexdigest() == SHA256
    again = torch.zeros(3674160, dtype=torch.uint8, device=dev())
    lib = _lib.load()
    _lib.check(lib.cube_distance_table_build(2, ctypes.c_void_p(again.data_ptr()),
                                             ctypes.c_void_p(torch.cuda.current_stream(dev()).cuda_stream)), "build")
    assert torch.equal(again, t)


def test_distance_matches_the_oracle(table):
    from rubiks_cube_solver_b200 import ops
    states = _scrambles(1 << 20, 1)
    got = ops.distance(2, states)
    assert got.shape == (1 << 20,) and got.dtype == torch.uint8
    want = D.distance_2(table, states.cpu().numpy())
    assert (got.cpu().numpy() == want).all()
    assert set(np.unique(want).tolist()) == set(range(15))
    for n in (0, 1, 31, 257, 1000):                                     # ragged: a block of 256 rows + 1
        out = ops.distance(2, states[:n])
        assert out.shape == (n,) and (out.cpu().numpy() == want[:n]).all()
    out = torch.empty(1 << 20, dtype=torch.uint8, device=dev())
    assert ops.distance(2, states, out=out) is out and (out.cpu().numpy() == want).all()


def test_garbage_rows_are_unreachable_and_outputs_stay_in_bounds(table):
    from rubiks_cube_solver_b200 import _lib, ops
    rows = _garbage(2)
    n = len(rows)
    want_d = D.distance_2(table, rows)
    assert (want_d[:4000] == 255).all() and (want_d[4000:] != 255).all()
    states = torch.from_numpy(rows).to(dev())
    lib, table_d = _lib.load(), ops.distance_table(dev())
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev()).cuda_stream)
    want_a, want_l = D.solve_optimal_2(table, rows)
    assert (want_l[:4000] == 255).all() and (want_a[:4000] == 12).all()
    for offset in (0, 3):                                                 # byte outputs may start anywhere
        raw_d, dist, lo_d = _guarded(n, offset)
        raw_a, acts, lo_a = _guarded(n * 14, offset)
        raw_l, length, lo_l = _guarded(n, offset + 1)
        _lib.check(lib.cube_distance(2, ctypes.c_void_p(table_d.data_ptr()), ctypes.c_void_p(states.data_ptr()), n,
                                     ctypes.c_void_p(dist.data_ptr()), stream), "cube_distance")
        _lib.check(lib.cube_solve_optimal(2, ctypes.c_void_p(table_d.data_ptr()), ctypes.c_void_p(states.data_ptr()), n,
                                          ctypes.c_void_p(acts.data_ptr()), ctypes.c_void_p(length.data_ptr()), stream),
                   "cube_solve_optimal")
        torch.cuda.synchronize()
        assert _guards_intact(raw_d, lo_d, n) and _guards_intact(raw_a, lo_a, n * 14) and _guards_intact(raw_l, lo_l, n)
        assert (dist.cpu().numpy() == want_d).all()
        assert (acts.view(n, 14).cpu().numpy() == want_a).all() and (length.cpu().numpy() == want_l).all()


def test_solve_optimal_matches_the_oracle_and_solves(table):
    from rubiks_cube_solver_b200 import ops
    states = _scrambles(200000, 3)
    actions, length = ops.solve_optimal(2, states)
    assert actions.shape == (200000, 14) and length.shape == (200000,)
    want_a, want_l = D.solve_optimal_2(table, states.cpu().numpy())
    assert (actions.cpu().numpy() == want_a).all() and (length.cpu().numpy() == want_l).all()
    assert torch.equal(length, ops.distance(2, states))
    end, solved, _ = ops.walk(2, states, actions)
    assert bool(solved.all())
    for n in (0, 1, 31, 129):                                             # ragged: a block of 128 rows + 1
        a, l = ops.solve_optimal(2, states[:n])
        assert (a.cpu().numpy() == want_a[:n]).all() and (l.cpu().numpy() == want_l[:n]).all()


def test_3x3x3_raises_not_implemented():
    from rubiks_cube_solver_b200 import ops
    states = ops.solved_states(3, 4, dev())
    with pytest.raises(NotImplementedError):
        ops.distance(3, states)
    with pytest.raises(NotImplementedError):
        ops.solve_optimal(3, states)


class DeepCube222(torch.nn.Module):
    """Layer shapes of model.py:7-29 for the reference's shipped 2x2x2 checkpoint (147-512-128-{64-6, 64-1}, ELU)."""

    def __init__(self, g):
        super().__init__()
        nn = torch.nn
        self.encoder_net = nn.Sequential(nn.Flatten(), nn.Linear(147, 512), nn.ELU(), nn.Linear(512, 128), nn.ELU())
        self.policy_net = nn.Sequential(nn.Linear(128, 64), nn.ELU(), nn.Linear(64, 6))
        self.value_net = nn.Sequential(nn.Linear(128, 64), nn.ELU(), nn.Linear(64, 1))
        self.load_state_dict({k[2:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("w:")})
        self.eval()

    def forward(self, x):
        h = self.encoder_net(x)
        return self.value_net(h), self.policy_net(h)


def _gap_stats(depths, solved, steps, dist):
    """optimal_gap's statistics, restated on the CPU."""
    out = []
    for i, d in enumerate(depths):
        s, t, k = solved[i], steps[i].astype(np.int64), dist[i].astype(np.int64)
        keep = s & (k > 0)
        out.append(dict(depth=int(d), solved_pct=float(s.mean()) * 100.0, mean_distance=float(k.mean()),
                        mean_steps=float(t[s].mean()) if s.any() else float("nan"),
                        mean_excess=float((t - k)[keep].mean()) if keep.any() else float("nan")))
    return out


def test_optimal_gap_with_the_reference_checkpoint(table):
    """rollout.optimal_gap at the golden depths and seeds equals the statistics of the recorded episodes
    (steps_plain / solved_plain) against the oracle's distances.  fp32 GEMMs on the GPU may order two nearly equal
    logits differently from the CPU (tests/test_pin222.py allows a handful of episodes for that), so the exact
    comparison with the recording is made when the GPU's own episodes reproduce it; optimal_gap always equals the
    statistics of the GPU's own episodes."""
    from rubiks_cube_solver_b200 import rollout
    g = np.load(os.path.join(HERE, "golden", "pin222.npz"))
    model = DeepCube222(g).cuda()
    seeds, depths = [int(s) for s in g["seeds"]], [int(d) for d in g["depths"]]
    max_t = int(g["max_timesteps"])
    gap = rollout.optimal_gap(model, seeds, depths, max_timesteps=max_t)
    starts = np.stack([O.scramble(2, np.random.RandomState(s).randint(6, size=(1, d)))[0] for d in depths for s in seeds])
    dist = D.distance_2(table, starts).reshape(len(depths), len(seeds))
    res = rollout.greedy_solve(model, 2, rollout.reference_scrambles(2, seeds, depths), max_timesteps=max_t)
    solved = res["solved"].cpu().numpy().reshape(dist.shape)
    steps = res["steps"].cpu().numpy().reshape(dist.shape)
    assert _nan_equal(gap, _gap_stats(depths, solved, steps, dist))
    golden = _gap_stats(depths, g["solved_plain"], g["steps_plain"], dist)
    if (solved == g["solved_plain"]).all() and (steps == g["steps_plain"]).all():
        assert _nan_equal(gap, golden)
    else:
        assert [r["mean_distance"] for r in gap] == [r["mean_distance"] for r in golden]
    for r in gap:
        assert r["mean_excess"] >= 0 and r["mean_steps"] >= 1
    model.cpu()


def _nan_equal(a, b):
    def key(rows):
        return [{k: ("nan" if isinstance(v, float) and v != v else v) for k, v in r.items()} for r in rows]
    return key(a) == key(b)
