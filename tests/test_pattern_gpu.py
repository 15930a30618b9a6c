"""The 3x3x3 pattern databases on the device (csrc/pattern.cu): the BFS build against the digests the CPU suite pins
for the emulated build, the bound and the bounded IDA* solve bit for bit against the kernels' per-state code run on
the CPU (tests/host_emul/pattern_emul.cpp) over the device-built tables, outputs at odd offsets between guard bytes,
and rollout.optimal_gap for the 3x3x3."""
import ctypes
import hashlib
import os
import subprocess

import numpy as np
import pytest
import torch

from oracle import pattern_np as P
from test_pattern_cpu import SHA256, emul_bound, emul_solve, garbage

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


def dev():
    return torch.device("cuda", 0)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream(dev()).cuda_stream)


@pytest.fixture(scope="module")
def emul(tmp_path_factory):
    lib_path = str(tmp_path_factory.mktemp("pattern_emul") / "libpattern_emul.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-pthread", "-w", "-o", lib_path,
                           os.path.join(HERE, "host_emul", "pattern_emul.cpp")])
    lib = ctypes.CDLL(lib_path)
    vp, ll, ci = ctypes.c_void_p, ctypes.c_longlong, ctypes.c_int
    lib.emul_pat3_bound.argtypes = [vp, vp, ll, vp, vp]
    lib.emul_pat3_solve.argtypes = [vp, vp, ll, ci, ll, vp, vp, vp, vp]
    return lib


@pytest.fixture(scope="module")
def host_tables():
    from rubiks_cube_solver_b200 import ops
    return ops.pattern_tables(dev()).cpu().numpy()


def _scrambles(n, seed, max_depth):
    """n sticker rows scrambled on the device, depths 0..max_depth (shorter rows padded with the no-op index)."""
    from rubiks_cube_solver_b200 import ops
    rng = np.random.RandomState(seed)
    moves = rng.randint(12, size=(n, max_depth)).astype(np.uint8)
    moves[np.arange(max_depth)[None, :] >= rng.randint(0, max_depth + 1, size=(n, 1))] = 12
    states, _, _ = ops.scramble(3, torch.from_numpy(moves).to(dev()), want_flags=False)
    return states


def _guarded(n_bytes, offset=0, guard=4096, fill=0xA5):
    """A device buffer with `guard` canary bytes on both sides of the payload, which starts `offset` bytes past a
    16-byte boundary."""
    raw = torch.full((guard + 16 + n_bytes + guard,), fill, dtype=torch.uint8, device=dev())
    lo = guard + (-(raw.data_ptr() + guard)) % 16 + offset
    return raw, raw[lo:lo + n_bytes], lo


def _guards_intact(raw, lo, n_bytes, fill=0xA5):
    return bool((raw[:lo] == fill).all()) and bool((raw[lo + n_bytes:] == fill).all())


def test_device_build_matches_the_pinned_digests():
    from rubiks_cube_solver_b200 import _lib, ops
    t = ops.pattern_tables(dev())
    assert t.dtype == torch.uint8 and t.shape == (P.TABLES_BYTES,) and ops.pattern_tables(dev()) is t      # cached
    raw, again, lo = _guarded(P.TABLES_BYTES, fill=0x5A)
    _lib.check(_lib.load().cube_pattern_tables_build(3, _ptr(again), _stream()), "cube_pattern_tables_build")
    torch.cuda.synchronize()
    assert _guards_intact(raw, lo, P.TABLES_BYTES, fill=0x5A) and torch.equal(again, t)
    got = t.cpu().numpy()
    for s in range(3):
        assert hashlib.sha256(got[P.OFFSETS[s]:P.OFFSETS[s] + P.ENTRIES[s]].tobytes()).hexdigest() == SHA256[s]


def test_bound_matches_the_emulation(emul, host_tables):
    from rubiks_cube_solver_b200 import _lib, ops
    bad = np.concatenate(garbage(7, 2000))
    rows = torch.cat([_scrambles(1 << 20, 1, 30), torch.from_numpy(bad).to(dev())]).contiguous()
    n = rows.shape[0]
    host_rows = rows.cpu().numpy()
    want_b, want_p = emul_bound(emul, host_tables, host_rows)
    assert (want_b[-len(bad):] == 255).all() and (want_b[:-len(bad)] != 255).all()
    assert set(np.unique(want_b[:-len(bad)]).tolist()) >= set(range(0, 13))
    b = ops.distance_bound(3, rows)
    b2, p2 = ops.distance_bound(3, rows, parts=True)
    assert (b.cpu().numpy() == want_b).all() and (b2.cpu().numpy() == want_b).all() and (p2.cpu().numpy() == want_p).all()
    for m in (0, 1, 127, 129, 1000):                                     # ragged: a block of 128 rows + 1
        assert (ops.distance_bound(3, rows[:m].contiguous()).cpu().numpy() == want_b[:m]).all()
    lib, tables = _lib.load(), ops.pattern_tables(dev())
    for offset in (0, 3):                                                # byte outputs may start anywhere
        raw_b, out_b, lo_b = _guarded(n, offset)
        raw_p, out_p, lo_p = _guarded(3 * n, offset + 1)
        _lib.check(lib.cube_distance_bound(3, _ptr(tables), _ptr(rows), n, _ptr(out_b), _ptr(out_p), _stream()),
                   "cube_distance_bound")
        torch.cuda.synchronize()
        assert _guards_intact(raw_b, lo_b, n) and _guards_intact(raw_p, lo_p, 3 * n)
        assert (out_b.cpu().numpy() == want_b).all() and (out_p.view(n, 3).cpu().numpy() == want_p).all()


def test_solve_matches_the_emulation_and_solves(emul, host_tables):
    from rubiks_cube_solver_b200 import _lib, ops
    bad = np.concatenate(garbage(8, 30))
    rows = torch.cat([_scrambles(4096, 2, 14), torch.from_numpy(bad).to(dev())]).contiguous()
    n, max_len, budget = rows.shape[0], 14, 1 << 17                       # the budget cuts some deep rows
    want_a, want_l, want_lo, want_n = emul_solve(emul, host_tables, rows.cpu().numpy(), max_len, budget)
    assert (want_l[-len(bad):] == 255).all() and (want_lo[-len(bad):] == 255).all()
    assert (want_l[:-len(bad)] != 255).mean() > 0.5 and (want_n == budget).any()
    a, l, lo, nodes = ops.solve_bounded(3, rows, max_length=max_len, max_nodes=budget, want_nodes=True)
    assert (a.cpu().numpy() == want_a).all() and (l.cpu().numpy() == want_l).all()
    assert (lo.cpu().numpy() == want_lo).all() and (nodes.cpu().numpy() == want_n).all()
    a3, l3, lo3 = ops.solve_bounded(3, rows, max_length=max_len, max_nodes=budget)
    assert torch.equal(a3, a) and torch.equal(l3, l) and torch.equal(lo3, lo)
    proven = l != 255
    _, solved, _ = ops.walk(3, rows[proven].contiguous(), a[proven].contiguous())
    assert bool(solved.all())
    lib, tables = _lib.load(), ops.pattern_tables(dev())
    for offset in (0, 5):
        raw_a, out_a, lo_a = _guarded(n * max_len, offset)
        raw_l, out_l, lo_l = _guarded(n, offset + 1)
        raw_o, out_o, lo_o = _guarded(n, offset + 2)
        raw_n, out_n, lo_n = _guarded(8 * n)
        _lib.check(lib.cube_solve_bounded(3, _ptr(tables), _ptr(rows), n, max_len, budget, _ptr(out_a), _ptr(out_l),
                                          _ptr(out_o), _ptr(out_n), _stream()), "cube_solve_bounded")
        torch.cuda.synchronize()
        assert _guards_intact(raw_a, lo_a, n * max_len) and _guards_intact(raw_l, lo_l, n)
        assert _guards_intact(raw_o, lo_o, n) and _guards_intact(raw_n, lo_n, 8 * n)
        assert (out_a.view(n, max_len).cpu().numpy() == want_a).all() and (out_l.cpu().numpy() == want_l).all()
        assert (out_o.cpu().numpy() == want_lo).all() and (out_n.view(torch.int64).cpu().numpy() == want_n).all()
    a0, l0, lo0 = ops.solve_bounded(3, rows[:0].contiguous())
    assert a0.shape == (0, 14) and l0.shape == (0,) and lo0.shape == (0,)


def test_2x2x2_raises_not_implemented():
    from rubiks_cube_solver_b200 import ops
    states = ops.solved_states(2, 4, dev())
    with pytest.raises(NotImplementedError):
        ops.distance_bound(2, states)
    with pytest.raises(NotImplementedError):
        ops.solve_bounded(2, states)


class SmallDeepCube(torch.nn.Module):
    """DeepCube's layout (model.py:7-29) at a small width, random weights: a policy that solves few cubes."""

    def __init__(self):
        super().__init__()
        nn = torch.nn
        torch.manual_seed(0)
        self.encoder_net = nn.Sequential(nn.Flatten(), nn.Linear(480, 64), nn.ELU())
        self.policy_net = nn.Linear(64, 12)
        self.value_net = nn.Linear(64, 1)

    def forward(self, x):
        h = self.encoder_net(x)
        return self.value_net(h), self.policy_net(h)


def test_optimal_gap_3x3x3(host_tables):
    from rubiks_cube_solver_b200 import ops, rollout
    model = SmallDeepCube().cuda()
    seeds, depths = list(range(0, 160, 10)), [1, 2, 3, 5, 8]
    gap = rollout.optimal_gap(model, seeds, depths, max_timesteps=20, cube_size=3)
    keys = {"depth", "solved_pct", "mean_distance", "mean_steps", "mean_excess", "proven_pct", "mean_lower_bound"}
    assert [r["depth"] for r in gap] == depths and all(set(r) == keys for r in gap)
    start, _, _ = ops.scramble(3, rollout.reference_scrambles_device(3, seeds, depths), want_flags=False)
    _, length, lower = ops.solve_bounded(3, start)
    length = length.cpu().numpy().reshape(len(depths), len(seeds)).astype(np.int64)
    lower = lower.cpu().numpy().reshape(len(depths), len(seeds)).astype(np.int64)
    for i, r in enumerate(gap):
        assert r["proven_pct"] == 100.0                                  # depth <= 8: always within the budget
        assert r["mean_distance"] == float(length[i].mean()) and r["mean_lower_bound"] == float(lower[i].mean())
        assert 0.0 <= r["solved_pct"] <= 100.0 and r["mean_distance"] <= depths[i]
        assert r["mean_excess"] != r["mean_excess"] or r["mean_excess"] >= 0
    model.cpu()
