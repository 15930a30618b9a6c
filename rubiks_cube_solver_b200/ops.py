"""Batched cube operators on CUDA tensors: thin, typed wrappers over the C ABI
(include/cube_b200.h).  PyTorch only supplies device memory and streams here.

Shapes: states ``[N, S]`` uint8 (S = 24 / 54), moves ``[N, depth]`` uint8,
one-hot ``[N, R, C]`` (7x21 / 20x24).  Every function launches asynchronously on
the current CUDA stream of the tensors' device and returns tensors on that device.
"""
import ctypes
import threading

import numpy as np
import torch

from . import _lib

N_STICKERS = {2: 24, 3: 54}
N_ACTIONS = {2: 6, 3: 12}
STATE_DIM = {2: (7, 21), 3: (20, 24)}                      # utils.py:162-186 get_env_config
ONEHOT_DTYPES = {torch.bfloat16: _lib.DTYPE_BF16, torch.float32: _lib.DTYPE_F32, torch.uint8: _lib.DTYPE_U8}
ENCODINGS = {"reference": _lib.ENCODING_REFERENCE, "exact": _lib.ENCODING_EXACT}


def _encoding(name):
    """"reference": the reference's one-hot tables as shipped (3x3x3 corners lossy, py333.py:140-180) -- the
    default, bit-exact against the reference.  "exact": the opt-in bijective 3x3x3 encoding (include/cube_b200.h),
    the only one `decode` can invert.  2x2x2 has a single encoding."""
    try:
        return ENCODINGS[name]
    except KeyError:
        raise ValueError("encoding must be 'reference' or 'exact', got %r" % (name,))


def _geom(cube_size):
    if cube_size not in (2, 3):
        raise NotImplementedError("cube_size must be 2 or 3")   # cube_env.py:43-44
    return N_STICKERS[cube_size], N_ACTIONS[cube_size], STATE_DIM[cube_size]


def _require_cuda(t, name, dtype=torch.uint8):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise TypeError("%s must be a CUDA tensor (this library has no CPU path)" % name)
    if t.dtype != dtype:
        raise TypeError("%s must have dtype %s, got %s" % (name, dtype, t.dtype))
    if not t.is_contiguous():
        raise ValueError("%s must be contiguous" % name)
    return t


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def sm_count():
    """SMs of the current device (C ABI cube_sm_count)."""
    return _lib.load().cube_sm_count()


def set_reserved_sms(n):
    """Leave n SMs free of the persistent kernels' CTAs (C ABI cube_set_reserved_sms), e.g. one for NCCL."""
    _lib.check(_lib.load().cube_set_reserved_sms(int(n)), "cube_set_reserved_sms")


def new_counters(device):
    """uint64[4] device counters: [solved, produced, bad actions, slow-path seeded rows] (kept as int64)."""
    return torch.zeros(4, dtype=torch.int64, device=device)


def solved_states(cube_size, n, device):
    """initState / initState_3 (py333.py:211-218): n solved cubes."""
    s, _, _ = _geom(cube_size)
    per = s // 6
    return torch.arange(6, dtype=torch.uint8, device=device).repeat_interleave(per).repeat(n, 1).contiguous()


def validate_actions(cube_size, actions):
    """Raise IndexError if any action index is >= A (cube_env.py:86,96).  Synchronises."""
    _geom(cube_size)
    actions = _require_cuda(actions, "actions")
    counters = new_counters(actions.device)
    with torch.cuda.device(actions.device):
        _lib.check(_lib.load().cube_validate_actions(cube_size, _ptr(actions), actions.numel(), _ptr(counters),
                                                     _stream(actions.device)), "cube_validate_actions")
    bad = int(counters[2].item())
    if bad:
        raise IndexError("%d action indices are out of range for cube_size %d" % (bad, cube_size))


def scramble(cube_size, moves, out=None, solved=None, reward=None, counters=None, want_flags=True):
    """Fused scramble from solved (C ABI cube_scramble).  Returns (states, solved, reward)."""
    s, _, _ = _geom(cube_size)
    moves = _require_cuda(moves, "moves")
    if moves.dim() != 2:
        raise ValueError("moves must be [N, depth]")
    n, depth = moves.shape
    dev = moves.device
    if out is None:
        out = torch.empty((n, s), dtype=torch.uint8, device=dev)
    _require_cuda(out, "out")
    if want_flags:
        if solved is None:
            solved = torch.empty(n, dtype=torch.uint8, device=dev)
        if reward is None:
            reward = torch.empty(n, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().cube_scramble(cube_size, _ptr(moves), n, depth, _ptr(out), _ptr(solved), _ptr(reward),
                                             _ptr(counters), _stream(dev)), "cube_scramble")
    return out, solved, reward


def scramble_step(cube_size, moves, actions, out=None, solved=None, reward=None, counters=None):
    """Scramble then one step, fused (C ABI cube_scramble_step): `reset` followed by `step(actions[i])` in one
    launch.  Returns (states, solved, reward) of the stepped cubes."""
    s, _, _ = _geom(cube_size)
    moves = _require_cuda(moves, "moves")
    actions = _require_cuda(actions, "actions")
    if moves.dim() != 2 or actions.numel() != moves.shape[0]:
        raise ValueError("moves must be [N, depth] and actions [N]")
    n, depth = moves.shape
    dev = moves.device
    if out is None:
        out = torch.empty((n, s), dtype=torch.uint8, device=dev)
    _require_cuda(out, "out")
    if solved is None:
        solved = torch.empty(n, dtype=torch.uint8, device=dev)
    if reward is None:
        reward = torch.empty(n, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().cube_scramble_step(cube_size, _ptr(moves), _ptr(actions), n, depth, _ptr(out), _ptr(solved),
                                                  _ptr(reward), _ptr(counters), _stream(dev)), "cube_scramble_step")
    return out, solved, reward


def prefixes_max_depth(cube_size):
    """Largest depth cube_scramble_prefixes takes (526 for 3x3x3, 1159 for 2x2x2)."""
    _geom(cube_size)
    return _lib.load().cube_scramble_prefixes_max_depth(cube_size)


def scramble_prefixes(cube_size, moves, out=None, want_solved=False, counters=None):
    """Every prefix of every scramble in one launch (C ABI cube_scramble_prefixes): returns
    (states [N, depth, S] uint8 cube-major, solved [N, depth] uint8 | None) -- the parents of an ADI batch in
    the order the reference appends its samples (cube_env.py:187-194)."""
    s, _, _ = _geom(cube_size)
    moves = _require_cuda(moves, "moves")
    if moves.dim() != 2:
        raise ValueError("moves must be [N, depth]")
    n, depth = moves.shape
    if depth > prefixes_max_depth(cube_size):
        raise ValueError("scramble_prefixes supports depth <= %d for cube_size %d" % (prefixes_max_depth(cube_size), cube_size))
    dev = moves.device
    if out is None:
        out = torch.empty((n, depth, s), dtype=torch.uint8, device=dev)
    _require_cuda(out, "out")
    if out.numel() != n * depth * s:
        raise ValueError("out must be [N, depth, %d]" % s)
    solved = torch.empty((n, depth), dtype=torch.uint8, device=dev) if want_solved else None
    with torch.cuda.device(dev):
        _lib.check(_lib.load().cube_scramble_prefixes(cube_size, _ptr(moves), n, depth, _ptr(out), _ptr(solved),
                                                      _ptr(counters), _stream(dev)), "cube_scramble_prefixes")
    return out, solved


def step(cube_size, states, actions, solved=None, reward=None, counters=None):
    """One transition in place (C ABI cube_step).  Returns (states, solved, reward)."""
    s, _, _ = _geom(cube_size)
    states = _require_cuda(states, "states")
    actions = _require_cuda(actions, "actions")
    n = states.shape[0]
    if states.shape != (n, s) or actions.numel() != n:
        raise ValueError("states must be [N, %d] and actions [N]" % s)
    dev = states.device
    if solved is None:
        solved = torch.empty(n, dtype=torch.uint8, device=dev)
    if reward is None:
        reward = torch.empty(n, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().cube_step(cube_size, _ptr(states), _ptr(actions), n, _ptr(solved), _ptr(reward),
                                         _ptr(counters), _stream(dev)), "cube_step")
    return states, solved, reward


def walk(cube_size, states, moves, out=None, solved=None, reward=None, counters=None):
    """`depth` transitions from given states (C ABI cube_walk); `out` may be `states`."""
    s, _, _ = _geom(cube_size)
    states = _require_cuda(states, "states")
    moves = _require_cuda(moves, "moves")
    n = states.shape[0]
    if moves.dim() == 1:
        moves = moves.view(n, 1)
    if states.shape != (n, s) or moves.shape[0] != n:
        raise ValueError("states must be [N, %d] and moves [N, depth]" % s)
    dev = states.device
    if out is None:
        out = torch.empty_like(states)
    if solved is None:
        solved = torch.empty(n, dtype=torch.uint8, device=dev)
    if reward is None:
        reward = torch.empty(n, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().cube_walk(cube_size, _ptr(states), _ptr(moves), n, moves.shape[1], _ptr(out),
                                         _ptr(solved), _ptr(reward), _ptr(counters), _stream(dev)), "cube_walk")
    return out, solved, reward


def is_solved(cube_size, states, counters=None):
    """Face uniformity + reward of resident states (C ABI cube_solved)."""
    s, _, _ = _geom(cube_size)
    states = _require_cuda(states, "states")
    n = states.shape[0]
    dev = states.device
    solved = torch.empty(n, dtype=torch.uint8, device=dev)
    reward = torch.empty(n, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().cube_solved(cube_size, _ptr(states), n, _ptr(solved), _ptr(reward), _ptr(counters),
                                           _stream(dev)), "cube_solved")
    return solved, reward


def encode(cube_size, states, dtype=torch.bfloat16, out=None, encoding="reference"):
    """One-hot network input [N, R, C] (C ABI cube_encode)."""
    s, _, (r, c) = _geom(cube_size)
    states = _require_cuda(states, "states")
    n = states.shape[0]
    dev = states.device
    if out is None:
        out = torch.empty((n, r, c), dtype=dtype, device=dev)
    _require_cuda(out, "out", dtype)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().cube_encode(cube_size, _ptr(states), n, _ptr(out), ONEHOT_DTYPES[dtype], _encoding(encoding),
                                           _stream(dev)), "cube_encode")
    return out


def expand(cube_size, states, dtype=torch.bfloat16, want_children=False, want_child_onehot=True,
           want_parent_onehot=False, child_onehot=None, counters=None, parent_onehot=None, solved=None, reward=None,
           want_reward=True, encoding="reference"):
    """All A children of every state (C ABI cube_expand).

    Returns dict(children [N,A,S] | None, child_onehot [N,A,R,C] | None,
    parent_onehot [N,R,C] | None, solved [N,A] uint8, reward [N,A] float32 | None).
    `child_onehot`, `parent_onehot`, `solved`, `reward` may be caller-owned output buffers (16-byte aligned
    slices of larger tensors are fine).
    """
    s, a, (r, c) = _geom(cube_size)
    states = _require_cuda(states, "states")
    n = states.shape[0]
    dev = states.device
    children = torch.empty((n, a, s), dtype=torch.uint8, device=dev) if want_children else None
    if want_child_onehot and child_onehot is None:
        child_onehot = torch.empty((n, a, r, c), dtype=dtype, device=dev)
    if child_onehot is not None:
        _require_cuda(child_onehot, "child_onehot", dtype)
        if child_onehot.numel() != n * a * r * c:
            raise ValueError("child_onehot must be [N, %d, %d, %d]" % (a, r, c))
    if want_parent_onehot and parent_onehot is None:
        parent_onehot = torch.empty((n, r, c), dtype=dtype, device=dev)
    if parent_onehot is not None:
        _require_cuda(parent_onehot, "parent_onehot", dtype)
        if parent_onehot.numel() != n * r * c:
            raise ValueError("parent_onehot must be [N, %d, %d]" % (r, c))
    if solved is None:
        solved = torch.empty((n, a), dtype=torch.uint8, device=dev)
    _require_cuda(solved, "solved")
    if reward is None and want_reward:
        reward = torch.empty((n, a), dtype=torch.float32, device=dev)
    if reward is not None:
        _require_cuda(reward, "reward", torch.float32)
    if solved.numel() != n * a or (reward is not None and reward.numel() != n * a):
        raise ValueError("solved / reward must be [N, %d]" % a)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().cube_expand(cube_size, _ptr(states), n, _ptr(children), _ptr(child_onehot),
                                           _ptr(parent_onehot), ONEHOT_DTYPES[dtype], _encoding(encoding), _ptr(solved),
                                           _ptr(reward), _ptr(counters), _stream(dev)), "cube_expand")
    return dict(children=children, child_onehot=child_onehot, parent_onehot=parent_onehot, solved=solved,
                reward=reward)


def key_bytes(cube_size):
    """Bytes of a compact code row (cube_expand_codes): the R column indices, zero-padded to whole words."""
    return (STATE_DIM[cube_size][0] + 3) & ~3


def expand_codes(cube_size, states, parent_dtype=None, want_children=False, counters=None, want_reward=True,
                 encoding="reference"):
    """All A children of every state with COMPACT CODES instead of one-hot rows (C ABI cube_expand_codes):
    code[row] = column of the 1 of that one-hot row = `onehot.argmax(-1)`, zero-padded to key_bytes.

    Returns dict(child_codes [N,A,KEY] uint8, parent_codes [N,KEY] uint8, parent_onehot [N,R,C] of
    `parent_dtype` | None, children [N,A,S] | None, solved [N,A] uint8, reward [N,A] float32)."""
    s, a, (r, c) = _geom(cube_size)
    states = _require_cuda(states, "states")
    n, dev, key = states.shape[0], states.device, key_bytes(cube_size)
    children = torch.empty((n, a, s), dtype=torch.uint8, device=dev) if want_children else None
    child_codes = torch.empty((n, a, key), dtype=torch.uint8, device=dev)
    parent_codes = torch.empty((n, key), dtype=torch.uint8, device=dev)
    parent_onehot = torch.empty((n, r, c), dtype=parent_dtype, device=dev) if parent_dtype is not None else None
    solved = torch.empty((n, a), dtype=torch.uint8, device=dev)
    reward = torch.empty((n, a), dtype=torch.float32, device=dev) if want_reward else None
    with torch.cuda.device(dev):
        _lib.check(_lib.load().cube_expand_codes(
            cube_size, _ptr(states), n, _ptr(children), _ptr(child_codes), _ptr(parent_codes), _ptr(parent_onehot),
            ONEHOT_DTYPES[parent_dtype] if parent_dtype is not None else _lib.DTYPE_U8, _encoding(encoding), _ptr(solved),
            _ptr(reward), _ptr(counters), _stream(dev)), "cube_expand_codes")
    return dict(child_codes=child_codes, parent_codes=parent_codes, parent_onehot=parent_onehot, children=children,
                solved=solved, reward=reward)


def moves_from_seeds(cube_size, seeds, depth, device=None, counters=None):
    """moves[i] = np.random.RandomState(seeds[i]).randint(A, size=depth) for every seed, drawn on the
    device (C ABI cube_moves_from_seeds): the scramble of reset(seed, depth), cube_env.py:62-65.
    seeds: ints in [0, 2**32) (sequence or tensor).  Returns uint8 [N, depth] on the device.
    counters[3] (new_counters) += rows that needed more than 227 raw draws (K0's slow path)."""
    _geom(cube_size)
    if not isinstance(seeds, torch.Tensor):
        seeds = torch.tensor([int(s) for s in seeds], dtype=torch.int64)
    seeds = seeds.to(torch.int64).reshape(-1)
    if seeds.numel() and (int(seeds.min()) < 0 or int(seeds.max()) >= 2 ** 32):
        raise ValueError("seeds must be in [0, 2**32): larger seeds take NumPy's init_by_array path")
    if depth < 0 or depth > 128:
        raise ValueError("moves_from_seeds supports 0 <= depth <= 128")
    if device is None:
        device = seeds.device if seeds.is_cuda else torch.device("cuda", torch.cuda.current_device())
    dev = torch.device(device)
    n = seeds.numel()
    s64 = seeds.to(dev)
    packed = torch.where(s64 >= 2 ** 31, s64 - 2 ** 32, s64).to(torch.int32).contiguous()      # the same 32 bits
    moves = torch.empty((n, depth), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().cube_moves_from_seeds(cube_size, _ptr(packed), n, depth, _ptr(moves), _ptr(counters),
                                                     _stream(dev)), "cube_moves_from_seeds")
    return moves


def adi_targets(cube_size, child_values, child_solved, parent_values, scramble_count, temperature):
    """ADI targets of cube_env.py:239-252 for a batch (C ABI cube_adi_targets).

    child_values float32 [P, A] = V(child); child_solved uint8 [P, A]; parent_values float32 [P];
    scramble_count int32 [P].  Returns (target_value float32 [P], target_policy int64 [P],
    error float64 [P]).  The weights k ** (-temperature) are computed here with Python's float power,
    exactly as the reference does, and looked up on the device."""
    _, a, _ = _geom(cube_size)
    child_values = _require_cuda(child_values.float().contiguous(), "child_values", torch.float32)
    p = child_values.shape[0]
    dev = child_values.device
    child_solved = _require_cuda(child_solved.contiguous(), "child_solved", torch.uint8)
    parent_values = _require_cuda(parent_values.float().contiguous(), "parent_values", torch.float32)
    scramble_count = scramble_count.to(device=dev, dtype=torch.int32).contiguous()
    if child_values.shape != (p, a) or child_solved.shape != (p, a) or parent_values.numel() != p or scramble_count.numel() != p:
        raise ValueError("adi_targets: shapes must be [P, %d], [P, %d], [P], [P]" % (a, a))
    kmax = int(scramble_count.max().item()) if p else 0
    table = [0.0] + [k ** (-1 * temperature) for k in range(1, kmax + 1)]          # cube_env.py:247
    weight = torch.tensor(table, dtype=torch.float64, device=dev)
    tv = torch.empty(p, dtype=torch.float32, device=dev)
    tp = torch.empty(p, dtype=torch.int32, device=dev)
    err = torch.empty(p, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.load().cube_adi_targets(cube_size, _ptr(child_values), _ptr(child_solved), _ptr(parent_values),
                                                _ptr(scramble_count), _ptr(weight), len(table), p, _ptr(tv), _ptr(tp),
                                                _ptr(err), _stream(dev)), "cube_adi_targets")
    return tv, tp.long(), err


def decode(cube_size, onehot, encoding="reference"):
    """One-hot -> sticker rows (C ABI cube_decode): [N, 7, 21] -> [N, 24] for 2x2x2; for 3x3x3 only the opt-in
    exact encoding has an inverse ([N, 20, 24] -> [N, 54]) -- with the reference's lossy table this raises
    NotImplementedError exactly like cube_env.py:171-172."""
    s, _, (r, c) = _geom(cube_size)
    enc = _encoding(encoding)
    if cube_size == 3 and enc != _lib.ENCODING_EXACT:
        raise NotImplementedError("3x3x3 decode is not implemented in the reference (cube_env.py:171-172): its corner "
                                  "encoding is lossy; encode and decode with encoding='exact'")
    if not onehot.is_cuda or onehot.dtype not in ONEHOT_DTYPES or not onehot.is_contiguous():
        raise TypeError("onehot must be a contiguous CUDA tensor of dtype bf16, f32 or u8")
    n = onehot.shape[0]
    if onehot.numel() != n * r * c:
        raise ValueError("onehot must be [N, %d, %d]" % (r, c))
    out = torch.empty((n, s), dtype=torch.uint8, device=onehot.device)
    with torch.cuda.device(onehot.device):
        _lib.check(_lib.load().cube_decode(cube_size, _ptr(onehot), ONEHOT_DTYPES[onehot.dtype], enc, n, _ptr(out),
                                           _stream(onehot.device)), "cube_decode")
    return out


_distance_tables = {}
_distance_lock = threading.Lock()


def distance_table(device=None):
    """The exact 2x2x2 distance table (C ABI cube_distance_table_build): uint8 [3674160], the quarter-turn
    distance of every rank (layout in include/cube_b200.h).  Built on the device the first time it is asked for
    there, then cached per device; treat it as read-only."""
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if dev.type != "cuda":
        raise TypeError("distance_table lives on a CUDA device (this library has no CPU path)")
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    with _distance_lock:
        table = _distance_tables.get(dev.index)
        if table is None:
            lib = _lib.load()
            table = torch.empty(_distance_entries(2), dtype=torch.uint8, device=dev)
            with torch.cuda.device(dev):
                _lib.check(lib.cube_distance_table_build(2, _ptr(table), _stream(dev)), "cube_distance_table_build")
                torch.cuda.current_stream(dev).synchronize()              # once: callers on any stream may read it
            _distance_tables[dev.index] = table
    return table


def _distance_entries(cube_size):
    _geom(cube_size)
    entries = _lib.load().cube_distance_table_entries(cube_size)
    if entries < 0:
        _lib.check(entries, "cube_distance_table_entries")                # 3x3x3: NotImplementedError
    return entries


def _distance_rows(cube_size, states):
    _distance_entries(cube_size)
    states = _require_cuda(states, "states")
    n = states.shape[0]
    if states.shape != (n, N_STICKERS[cube_size]):
        raise ValueError("states must be [N, %d]" % N_STICKERS[cube_size])
    return states, n, distance_table(states.device)


def distance(cube_size, states, out=None):
    """Exact distance of every sticker row (C ABI cube_distance): uint8 [N], 255 for a row that is not a
    reachable state.  2x2x2 only (3x3x3 raises NotImplementedError)."""
    states, n, table = _distance_rows(cube_size, states)
    dev = states.device
    if out is None:
        out = torch.empty(n, dtype=torch.uint8, device=dev)
    _require_cuda(out, "out")
    if out.numel() != n:
        raise ValueError("out must hold N = %d distances" % n)
    if n:
        with torch.cuda.device(dev):
            _lib.check(_lib.load().cube_distance(cube_size, _ptr(table), _ptr(states), n, _ptr(out), _stream(dev)),
                       "cube_distance")
    return out


def solve_optimal(cube_size, states):
    """An optimal solution of every row (C ABI cube_solve_optimal): returns (actions uint8 [N, 14] padded with the
    no-op index 12, length uint8 [N]); at every step the lowest action index whose child is one level closer.
    `walk(cube_size, states, actions)` ends solved for every reachable row; an unreachable row gets length 255
    and only no-ops.  2x2x2 only."""
    states, n, table = _distance_rows(cube_size, states)
    dev = states.device
    actions = torch.empty((n, _lib.DISTANCE_MAX_2), dtype=torch.uint8, device=dev)
    length = torch.empty(n, dtype=torch.uint8, device=dev)
    if n:
        with torch.cuda.device(dev):
            _lib.check(_lib.load().cube_solve_optimal(cube_size, _ptr(table), _ptr(states), n, _ptr(actions),
                                                      _ptr(length), _stream(dev)), "cube_solve_optimal")
    return actions, length


_pattern_tables = {}
_pattern_lock = threading.Lock()

# Per-row node budget of solve_bounded.  On seeded scrambles of depth 8 / 10 / 12 / 14 (4 096 each) the search needed
# at most 893 / 3 943 / 63 570 / 2 157 028 child states (tools/distance_333.py, profiles/r04_distance_333.json; B200,
# 1 000 W), so 4 Mi proves all of them with room to spare.  A row runs in one thread, which generated at least 0.45 M
# children per second there (2.16 M within the 4.76 s call): one row that exhausts 4 Mi holds a call about 9 s.
SOLVE_BOUNDED_MAX_NODES = 1 << 22


def _pattern_bytes(cube_size):
    _geom(cube_size)
    n = _lib.load().cube_pattern_tables_bytes(cube_size)
    if n < 0:
        _lib.check(n, "cube_pattern_tables_bytes")                        # 2x2x2: NotImplementedError
    return n


def pattern_tables(device=None):
    """The 3x3x3 pattern databases (C ABI cube_pattern_tables_build): uint8 [173335680], the corner table and the two
    6-edge tables (layout in include/cube_b200.h).  Built on the device the first time they are asked for there,
    then cached per device; treat them as read-only."""
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if dev.type != "cuda":
        raise TypeError("pattern_tables live on a CUDA device (this library has no CPU path)")
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    with _pattern_lock:
        tables = _pattern_tables.get(dev.index)
        if tables is None:
            lib = _lib.load()
            tables = torch.empty(_pattern_bytes(3), dtype=torch.uint8, device=dev)
            with torch.cuda.device(dev):
                _lib.check(lib.cube_pattern_tables_build(3, _ptr(tables), _stream(dev)), "cube_pattern_tables_build")
                torch.cuda.current_stream(dev).synchronize()              # once: callers on any stream may read them
            _pattern_tables[dev.index] = tables
    return tables


def _pattern_rows(cube_size, states):
    _pattern_bytes(cube_size)
    states = _require_cuda(states, "states")
    n = states.shape[0]
    if states.shape != (n, N_STICKERS[cube_size]):
        raise ValueError("states must be [N, %d]" % N_STICKERS[cube_size])
    return states, n, pattern_tables(states.device)


def distance_bound(cube_size, states, parts=False):
    """Admissible quarter-turn lower bound of every sticker row (C ABI cube_distance_bound): uint8 [N], 255 for a
    row that is not a reachable state; with parts=True also the corner, edges-A and edges-B values, uint8 [N, 3].
    3x3x3 only (2x2x2 raises NotImplementedError: use `distance`)."""
    states, n, tables = _pattern_rows(cube_size, states)
    dev = states.device
    bound = torch.empty(n, dtype=torch.uint8, device=dev)
    p = torch.empty((n, 3), dtype=torch.uint8, device=dev) if parts else None
    if n:
        with torch.cuda.device(dev):
            _lib.check(_lib.load().cube_distance_bound(cube_size, _ptr(tables), _ptr(states), n, _ptr(bound), _ptr(p),
                                                       _stream(dev)), "cube_distance_bound")
    return (bound, p) if parts else bound


def solve_bounded(cube_size, states, max_length=14, max_nodes=SOLVE_BOUNDED_MAX_NODES, want_nodes=False):
    """Proven optimal solutions within a budget (C ABI cube_solve_bounded): IDA* over the pattern-database bound, one
    thread per row.  Returns (actions uint8 [N, max_length] padded with the no-op index 12, length uint8 [N] = the
    optimal length or 255 where it was not proven, lower uint8 [N] = the best proven lower bound[, nodes int64 [N]]).
    A row is unproven when the search reached max_length (lower > max_length) or generated max_nodes children;
    `walk(cube_size, states, actions)` ends solved for every proven row.  3x3x3 only."""
    if not 0 <= max_length <= _lib.SOLVE_BOUNDED_MAX_LENGTH:
        raise ValueError("max_length must be in 0..%d" % _lib.SOLVE_BOUNDED_MAX_LENGTH)
    if max_nodes < 0:
        raise ValueError("max_nodes must be >= 0")
    states, n, tables = _pattern_rows(cube_size, states)
    dev = states.device
    actions = torch.empty((n, max_length), dtype=torch.uint8, device=dev)
    length = torch.empty(n, dtype=torch.uint8, device=dev)
    lower = torch.empty(n, dtype=torch.uint8, device=dev)
    nodes = torch.empty(n, dtype=torch.int64, device=dev) if want_nodes else None
    if n:
        with torch.cuda.device(dev):
            _lib.check(_lib.load().cube_solve_bounded(cube_size, _ptr(tables), _ptr(states), n, max_length, max_nodes,
                                                      _ptr(actions), _ptr(length), _ptr(lower), _ptr(nodes),
                                                      _stream(dev)), "cube_solve_bounded")
    return (actions, length, lower, nodes) if want_nodes else (actions, length, lower)


class HostCube(object):
    """One cube per call through host (NumPy) buffers -- C ABI cube_env_host_*: the per-call path of the
    drop-in CubeEnv (reset / step / get_obs, cube_env.py:56-147).  Two launches and one stream
    synchronisation per call, no copy calls (the kernels work on a mapped pinned page).  Bound to one
    device; not thread-safe (use one per thread, see `host_cube`)."""

    def __init__(self, cube_size, device=None, max_depth=1024):
        self.s, _, (r, c) = _geom(cube_size)
        self.shape = (r, c)
        self.cube_size, self.max_depth = cube_size, max_depth
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self._idx = dev.index if dev.index is not None else torch.cuda.current_device()
        handle = ctypes.c_void_p()
        lib = _lib.load()
        with torch.cuda.device(self._idx):
            _lib.check(lib.cube_env_host_create(cube_size, max_depth, ctypes.byref(handle)), "cube_env_host_create")
        self._h = handle
        self._step, self._scramble, self._encode = lib.cube_env_host_step, lib.cube_env_host_scramble, lib.cube_env_host_encode
        self._solved = ctypes.c_int(0)
        self._solved_ref = ctypes.byref(self._solved)

    def _run(self, fn, *args):
        if torch.cuda.current_device() != self._idx:
            with torch.cuda.device(self._idx):
                rc = fn(self._h, *args)
        else:
            rc = fn(self._h, *args)
        if rc:
            _lib.check(rc, fn.__name__)

    def step(self, stickers, action):
        """stickers: uint8 [S] NumPy array, action: int.  Returns (stickers uint8 [S], onehot uint8 [R, C], solved)."""
        out = np.empty(self.s, dtype=np.uint8)
        onehot = np.empty(self.shape, dtype=np.uint8)
        self._run(self._step, stickers.ctypes.data, int(action), out.ctypes.data, onehot.ctypes.data, self._solved_ref, None)
        return out, onehot, bool(self._solved.value)

    def scramble(self, moves):
        """moves: uint8 [depth] NumPy array applied to the solved cube.  Same returns as `step`."""
        if len(moves) > self.max_depth:
            raise ValueError("more than max_depth = %d moves" % self.max_depth)
        out = np.empty(self.s, dtype=np.uint8)
        onehot = np.empty(self.shape, dtype=np.uint8)
        self._run(self._scramble, moves.ctypes.data, len(moves), out.ctypes.data, onehot.ctypes.data, self._solved_ref, None)
        return out, onehot, bool(self._solved.value)

    def encode(self, stickers):
        onehot = np.empty(self.shape, dtype=np.uint8)
        self._run(self._encode, stickers.ctypes.data, onehot.ctypes.data, None)
        return onehot

    def close(self):
        if self._h:
            _lib.load().cube_env_host_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001 - interpreter shutdown
            pass


_host_cubes = threading.local()


def host_cube(cube_size, device_index):
    """The calling thread's HostCube for (cube_size, device): envs share it, so `copy.deepcopy(env)`
    (mcts.py:37,96,101) copies no handle."""
    cache = getattr(_host_cubes, "cache", None)
    if cache is None:
        cache = _host_cubes.cache = {}
    key = (cube_size, device_index)
    hc = cache.get(key)
    if hc is None:
        hc = cache[key] = HostCube(cube_size, torch.device("cuda", device_index))
    return hc


class HostScramblePipeline(object):
    """End-to-end fused scramble for host arrays (C ABI cube_pipeline_*): chunked H2D copy,
    kernel and D2H copy overlapped over a few streams.  Bound to one device."""

    def __init__(self, cube_size, depth, chunk_instances=1 << 20, n_stages=3, device=None):
        self.s, _, _ = _geom(cube_size)
        self.cube_size, self.depth = cube_size, depth
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        handle = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().cube_pipeline_create(cube_size, depth, chunk_instances, n_stages,
                                                        ctypes.byref(handle)), "cube_pipeline_create")
        self._h = handle

    def _outputs(self, n, states_out, solved, reward, want_solved, want_reward):
        if states_out is None:
            states_out = torch.empty((n, self.s), dtype=torch.uint8).pin_memory()
        if solved is None and want_solved:
            solved = torch.empty(n, dtype=torch.uint8).pin_memory()
        if reward is None and want_reward:
            reward = torch.empty(n, dtype=torch.float32).pin_memory()
        return states_out, solved, reward

    @staticmethod
    def _hp(t):
        return None if t is None else ctypes.c_void_p(t.data_ptr())

    def run(self, moves_host, states_out=None, solved=None, reward=None, want_solved=True, want_reward=True):
        """moves_host: CPU uint8 tensor [N, depth] (pinned for full overlap).  Returns CPU tensors
        (states, solved, reward) and the solved count; blocks until they are filled.  `want_reward=False`
        skips the reward array (4 of 59 bytes per instance on the way back: it is +-1 by `solved`)."""
        if moves_host.is_cuda or moves_host.dtype != torch.uint8 or not moves_host.is_contiguous():
            raise TypeError("moves_host must be a contiguous CPU uint8 tensor")
        n = moves_host.shape[0]
        if moves_host.shape != (n, self.depth):
            raise ValueError("moves_host must be [N, %d]" % self.depth)
        states_out, solved, reward = self._outputs(n, states_out, solved, reward, want_solved, want_reward)
        count = ctypes.c_int64(0)
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().cube_pipeline_scramble_host(
                self._h, ctypes.c_void_p(moves_host.data_ptr()), n, self._hp(states_out), self._hp(solved),
                self._hp(reward), ctypes.byref(count)), "cube_pipeline_scramble_host")
        return states_out, solved, reward, int(count.value)

    def reset(self, seeds_host, states_out=None, solved=None, reward=None, want_solved=True, want_reward=True):
        """Batched `reset(seed, depth)` (cube_env.py:50-69) for host arrays (C ABI cube_pipeline_reset_host):
        seeds_host is a CPU int32 / uint32-valued tensor [N] (the 32 bits of each seed); only 4 bytes per cube
        go to the device, the moves are drawn there.  Same returns as `run`."""
        if seeds_host.is_cuda or seeds_host.dtype != torch.int32 or not seeds_host.is_contiguous():
            raise TypeError("seeds_host must be a contiguous CPU int32 tensor (the seeds' 32 bits)")
        if not 1 <= self.depth <= 128:
            raise ValueError("seeded resets need 1 <= depth <= 128")
        n = seeds_host.numel()
        states_out, solved, reward = self._outputs(n, states_out, solved, reward, want_solved, want_reward)
        count = ctypes.c_int64(0)
        with torch.cuda.device(self.device):
            _lib.check(_lib.load().cube_pipeline_reset_host(
                self._h, ctypes.c_void_p(seeds_host.data_ptr()), n, self._hp(states_out), self._hp(solved),
                self._hp(reward), ctypes.byref(count)), "cube_pipeline_reset_host")
        return states_out, solved, reward, int(count.value)

    def close(self):
        if self._h:
            _lib.load().cube_pipeline_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001 - interpreter shutdown
            pass


class _HostBlock(object):
    def __init__(self, ptr):
        self.ptr = ptr

    def __del__(self):
        try:
            _lib.load().cube_host_free(self.ptr)
        except Exception:  # noqa: BLE001 - interpreter shutdown
            pass


def host_buffer(shape, dtype=torch.uint8):
    """A page-locked CPU tensor on 2 MiB transparent huge pages (C ABI cube_host_alloc) for the host arrays of
    `HostScramblePipeline`; freed when the tensor is garbage-collected."""
    shape = tuple(int(x) for x in (shape if isinstance(shape, (tuple, list)) else (shape,)))
    n = 1
    for x in shape:
        n *= x
    nbytes = max(1, n * torch.empty(0, dtype=dtype).element_size())
    ptr = ctypes.c_void_p()
    _lib.check(_lib.load().cube_host_alloc(nbytes, ctypes.byref(ptr)), "cube_host_alloc")
    block = _HostBlock(ptr)
    raw = (ctypes.c_uint8 * nbytes).from_address(ptr.value)
    t = torch.frombuffer(raw, dtype=torch.uint8, count=nbytes)
    t = t.view(dtype)[:n].view(shape)
    _host_blocks.append(block)
    return t


_host_blocks = []          # views of a buffer share its storage: the mappings live until release_host_buffers()


def release_host_buffers():
    """Free every buffer handed out by `host_buffer` (call when none of them is in use any more)."""
    del _host_blocks[:]
