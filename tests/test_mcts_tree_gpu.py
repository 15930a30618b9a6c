"""The batched MCTS tree kernels (cube_mcts_traverse, cube_mcts_update) in lock-step with the oracle's tree.

The tree kernels only ever see keys, values and policies, so this file supplies them itself and drives the two
entry points directly: per simulation one traversal, a comparison of everything it wrote with
oracle/mcts_ref.MCTSRef's traverse, then the leaf's children (oracle/cube_np), keys, value and policy, one
update, and a comparison of the WHOLE tree store -- every slot's key, child keys, done flags, P, W, N, L and
memoised child slot -- with the oracle's dict.  Every array of the tree store and every input and output of both
calls sits between guard bytes.

Keys are a function of the sticker row that both sides share: the production codes (`real`), a hash into a small
key space so that different cubes alias (`colliding`: overwrites of existing nodes, re-found keys, nodes that are
their own child, edges backed up twice on one path), and keys that differ only in their last 32-bit word or only
in their first byte.  The search constants and the optional inputs (sim_counter / n_active, an odd path_cap that
takes the update's byte path) vary across the cases, and coverage counters taken from the oracle show that the
paths each case targets really ran.  A second group runs the capacity flags and checks that those error paths
stay inside the caller's buffers."""
import ctypes
import random

import numpy as np
import pytest
import torch

from rubiks_cube_solver_b200 import _lib
from rubiks_cube_solver_b200.mcts_batch import BatchedMCTS, _Tree

from oracle import cube_np as O
from oracle import mcts_ref
from oracle import tables as T

pytestmark = pytest.mark.gpu
SIZES = (2, 3)
FILL = 0xA5
KEY = {2: 8, 3: 20}
B, NUM_SIM = 300, 40
# (cpuct, virtual_loss, value_min): the defaults; others; value_min above many backed-up values.  The way up always
# removes 150 (mcts.py:128), so a virtual loss below 150 leaves a visited edge with a negative L that grows with
# its visits: the reference's traversal then circles its own path for ever longer (virtual_loss = 7 gives paths of
# ~18 000 steps by the sixth simulation), so every set here keeps virtual_loss >= 150.
CONSTS = ((1.0, 150, -10.0), (0.37, 160, -3.5), (2.5, 1000, 0.25))
INACTIVE = (5, 17, 18, 131, 299)           # trees that never search: inside a warp, and the very last one


def dev():
    return torch.device("cuda", 0)


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


# ------------------------------------------------------------------ keys, values, policies
_W = np.random.RandomState(99).randint(1, 1 << 20, size=64).astype(np.int64)


def _hash(rows, mod):
    """A fixed linear hash of uint8 rows, reduced mod `mod` (< 2^32)."""
    rows = np.asarray(rows, dtype=np.int64)
    return (rows @ _W[:rows.shape[1]] * 2654435761 + 12345) % (1 << 61) % mod


def real_key(size, states):
    """The production key: the one-hot's column per row (argmax), the 2x2x2's padded to 8 bytes (BatchedMCTS._codes)."""
    cols = O.onehot_columns(size, states)
    out = np.zeros((len(states), KEY[size]), dtype=np.uint8)
    out[:, :cols.shape[1]] = cols
    return out


def make_key(mode, size):
    """key(states [n, S] uint8) -> [n, KEY] uint8 for each key mode."""
    kb = KEY[size]
    fixed = (np.arange(kb, dtype=np.int64) * 37 + 11).astype(np.uint8)

    def key(states):
        n = len(states)
        if mode == "real":
            return real_key(size, states)
        out = np.tile(fixed, (n, 1))
        if mode == "colliding":                       # ~ 2 * NUM_SIM keys: aliasing is everywhere, traversals still end
            h = _hash(states, 2 * NUM_SIM + 5)
            out[:, :] = (h[:, None] * 7 + np.arange(kb)[None, :]) % 256
        elif mode == "lastword":                      # distinct keys equal in every word but the last
            h = _hash(real_key(size, states), 1 << 32)
            out[:, -4:] = (h[:, None] >> (8 * np.arange(4))[None, :]) & 0xff
        else:                                          # "firstbyte": they differ in byte 0 only
            out[:, 0] = _hash(real_key(size, states), 251)
        return out
    return key


def value_policy(keys, a):
    """Deterministic functions of the leaf key: a dyadic value in [-2, 2] (never -0.0), positive float32 policies."""
    h = _hash(keys, 1 << 31)
    value = ((h % 33).astype(np.float32) - 16.0) / np.float32(8.0)
    ks = np.repeat(keys.astype(np.int64), a, axis=0)
    ks[:, 0] += np.tile(np.arange(1, a + 1), len(keys)) * 256
    hp = _hash(ks, 1 << 24).reshape(len(keys), a)
    policy = ((hp + 1).astype(np.float64) / 16777259.0).astype(np.float32)
    return value.astype(np.float32), policy


# ------------------------------------------------------------------ the oracle
class StickerEnv(object):
    """The env of MCTSRef over the oracle's sticker rows: step returns the sticker row as the observation."""

    def __init__(self, size, row):
        self.size, self.sim = size, row

    def __deepcopy__(self, memo):
        return StickerEnv(self.size, self.sim)                  # rows are never written in place

    def step(self, a):
        self.sim = self.sim[T.MOVE_DEFS[self.size][a]]
        k = T.N_STICKERS[self.size] // 6
        faces = self.sim.reshape(6, k)
        done = bool((faces == faces[:, :1]).all())
        return self.sim, (1.0 if done else -1.0), done, {}


class Draws(random.Random):
    """random.Random(seed) that counts its draws."""

    def __init__(self, seed):
        super().__init__(seed)
        self.n = 0

    def randint(self, a, b):
        self.n += 1
        return super().randint(a, b)


class KeyedRef(mcts_ref.MCTSRef):
    """MCTSRef with the test's key; keys and predictions of the batch are computed once per simulation."""

    def __init__(self, cache, predict, action_dim, consts, rng):
        cpuct, vl, vmin = consts
        super().__init__(predict, action_dim, loss_constant=vl, cpuct=cpuct, value_min=vmin, rng=rng)
        self.cache = cache

    def key(self, obs):
        return self.cache[np.ascontiguousarray(obs).tobytes()]


class OracleBatch(object):
    """B oracle trees driven one simulation at a time, with expected device arrays and coverage counters."""

    def __init__(self, size, mode, consts, roots, active, seeds, n_slots):
        self.size, self.A, self.kb, self.M = size, T.N_ACTIONS[size], KEY[size], n_slots
        self.key = make_key(mode, size)
        self.cache, self.pred = {}, {}
        self.roots = roots
        self.remember(roots)
        self.trees = [KeyedRef(self.cache, self.predict, self.A, consts, Draws(sd)) for sd in seeds]
        self.active = active.copy()
        self.slot_of = [dict() for _ in range(len(roots))]
        b, m, a, kb = len(roots), n_slots, self.A, self.kb

        def fill(shape, dtype):
            return np.full(int(np.prod(shape)) * np.dtype(dtype).itemsize, FILL, np.uint8).view(dtype).reshape(shape)
        self.E = dict(node_key=fill((b, m, kb), np.uint8), child_key=fill((b, m, a, kb), np.uint8),
                      child_done=fill((b, m, a), np.uint8), P=fill((b, m, a), np.float32), W=fill((b, m, a), np.float32),
                      N=fill((b, m, a), np.int32), L=fill((b, m, a), np.int32),
                      child_slot=np.full((b, m, a), 255, np.uint8), n_nodes=np.zeros(b, np.int32))
        self.cov = dict(overwrite=0, refound=0, self_child=0, bounce=0, path16=0, path32=0, solved=0, budget=0,
                        longest=0)

    def remember(self, rows):
        keys = self.key(rows)
        for r, k in zip(rows, keys):
            self.cache[r.tobytes()] = k.tobytes()
        return keys

    def predict(self, state):
        return self.pred[np.ascontiguousarray(state).tobytes()]

    def traverse(self):
        """MCTSRef.traverse of every active tree: expected path slots / actions / lengths, leaf rows, draws."""
        b = len(self.trees)
        self.walk = [None] * b
        plen = np.zeros(b, np.int32)
        leaf = self.roots.copy()
        for i in np.flatnonzero(self.active):
            t = self.trees[i]
            env = StickerEnv(self.size, self.roots[i])
            path, actions, cur = t.traverse(self.roots[i], env)
            self.walk[i] = (path, actions, cur, env)
            plen[i] = len(path)
            leaf[i] = cur
            for node, act in zip(path, actions):
                self.refresh_row(i, node)
            pairs = list(zip(path, actions))
            self.cov["bounce"] += len(set(pairs)) < len(pairs)
            self.cov["path16"] += len(path) > 16
            self.cov["path32"] += len(path) > 32
            self.cov["longest"] = max(self.cov["longest"], len(path))
        return plen, leaf

    def expected_path(self, i):
        path, actions = self.walk[i][:2]
        return [self.slot_of[i][k] for k in path], actions

    def update(self, sim, leaf):
        """Children, keys, value and policy of every leaf (batched), then expand + backpropagate + exit test of
        every active tree.  Returns the device inputs and {tree: action list} of the trees that solved."""
        children, done = O.expand(self.size, leaf)
        child_keys = self.remember(children.reshape(-1, children.shape[-1])).reshape(len(leaf), self.A, self.kb)
        leaf_keys = self.remember(leaf)
        value, policy = value_policy(leaf_keys, self.A)
        for r, v, p in zip(leaf, value, policy):
            self.pred[r.tobytes()] = (np.array([v], np.float32), p)
        solved = {}
        for i in np.flatnonzero(self.active):
            t = self.trees[i]
            path, actions, cur, env = self.walk[i]
            k = t.key(cur)
            if k in t.nodes:
                self.cov["overwrite"] += 1
            elif any(k in node[0] for node in t.nodes.values()):
                self.cov["refound"] += 1
            v = t.expand(cur, env)
            t.backpropagate(path, actions, v)
            if k not in self.slot_of[i]:
                self.slot_of[i][k] = len(self.slot_of[i])
            self.cov["self_child"] += k in t.nodes[k][0]
            for node in set(path) | {k}:
                self.refresh_row(i, node)
            self.refresh_memo(i)
            for j, d in enumerate(t.nodes[k][5]):
                if d:
                    solved[i] = actions + [j]
                    break
        for i in solved:
            self.active[i] = 0
        self.cov["solved"] += len(solved)
        if sim == NUM_SIM - 1:
            self.cov["budget"] += int(self.active.sum())
        return leaf_keys, child_keys, done.astype(np.uint8), value, policy, solved

    def refresh_row(self, i, k):
        s = self.slot_of[i][k]
        children, P, W, N, L, done = self.trees[i].nodes[k]
        E = self.E
        E["node_key"][i, s] = np.frombuffer(k, np.uint8)
        E["child_key"][i, s] = np.frombuffer(b"".join(children), np.uint8).reshape(self.A, self.kb)
        E["child_done"][i, s] = done
        E["P"][i, s] = P
        E["W"][i, s] = W
        E["N"][i, s] = N
        E["L"][i, s] = L
        E["n_nodes"][i] = len(self.slot_of[i])

    def refresh_memo(self, i):
        so = self.slot_of[i]
        for k, s in so.items():
            self.E["child_slot"][i, s] = [so.get(c, 255) for c in self.trees[i].nodes[k][0]]

    def rebuild(self, i):
        """The expected rows of tree i from scratch (checks the incremental bookkeeping)."""
        for k in self.trees[i].nodes:
            self.refresh_row(i, k)
        self.refresh_memo(i)


# ------------------------------------------------------------------ the device side
TREE_FIELDS = [name for name, _ in _Tree._fields_[4:]]


class DeviceTrees(object):
    """The tree store of B trees and every input / output of the two calls, each between canaries."""

    def __init__(self, size, n, n_slots, path_cap, rand_cap, with_counter):
        A, S, kb = T.N_ACTIONS[size], T.N_STICKERS[size], KEY[size]
        self.size, self.n, self.M, self.path_cap, self.rand_cap = size, n, n_slots, path_cap, rand_cap
        spec = dict(node_key=((n, n_slots, kb), torch.uint8), child_key=((n, n_slots, A, kb), torch.uint8),
                    child_done=((n, n_slots, A), torch.uint8), P=((n, n_slots, A), torch.float32),
                    W=((n, n_slots, A), torch.float32), N=((n, n_slots, A), torch.int32), L=((n, n_slots, A), torch.int32),
                    n_nodes=((n,), torch.int32), active=((n,), torch.uint8), root_state=((n, S), torch.uint8),
                    root_key=((n, kb), torch.uint8), rand_table=((n, rand_cap), torch.uint8), rand_ptr=((n,), torch.int32),
                    path_node=((n, path_cap), torch.uint8), path_action=((n, path_cap), torch.uint8),
                    path_len=((n,), torch.int32), leaf_state=((n, S), torch.uint8), flags=((1,), torch.int32),
                    child_slot=((n, n_slots, A), torch.uint8), sim_counter=((1,), torch.int32),
                    leaf_key=((n, kb), torch.uint8), child_key_new=((n, A, kb), torch.uint8),
                    child_done_new=((n, A), torch.uint8), value=((n,), torch.float32), policy=((n, A), torch.float32),
                    actions_out=((n, path_cap + 1), torch.int8), n_actions=((n,), torch.int32),
                    n_sims=((n,), torch.int32), n_active=((NUM_SIM,), torch.int32))
        self.g = {}
        for name, (shape, dtype) in spec.items():
            if name in ("sim_counter", "n_active") and not with_counter:
                continue
            g = Guarded(int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size(), dtype)
            g.view = g.view.view(shape)
            self.g[name] = g
        for name in ("n_nodes", "rand_ptr", "path_len", "flags", "n_actions"):
            self.g[name].view.zero_()
        self.g["child_slot"].view.fill_(255)
        self.g["actions_out"].view.fill_(-1)
        self.g["n_sims"].view.fill_(-7)
        if with_counter:
            self.g["sim_counter"].view.fill_(-1)
            self.g["n_active"].view.zero_()
        self.tree = _Tree(n, n_slots, path_cap, rand_cap,
                          *[self.g[f].view.data_ptr() if f in self.g else None for f in TREE_FIELDS])

    def __getitem__(self, name):
        return self.g[name].view

    def ptr(self, name):
        return self.g[name].view.data_ptr() if name in self.g else None

    def host(self, name):
        return self.g[name].view.cpu().numpy()

    def traverse(self, cpuct, vl):
        return self.lib().cube_mcts_traverse(self.size, ctypes.byref(self.tree), ctypes.c_float(cpuct), vl, _stream())

    def update(self, vmin, sim_index):
        p = self.ptr
        return self.lib().cube_mcts_update(self.size, ctypes.byref(self.tree), p("leaf_key"), p("child_key_new"),
                                           p("child_done_new"), p("value"), p("policy"), ctypes.c_float(vmin), sim_index,
                                           p("actions_out"), p("n_actions"), p("n_sims"), p("n_active"), _stream())

    @staticmethod
    def lib():
        return _lib.load()

    def upload(self, **arrays):
        for name, a in arrays.items():
            self.g[name].view.copy_(torch.from_numpy(np.ascontiguousarray(a)).view(self.g[name].view.dtype)
                                    .reshape(self.g[name].view.shape))

    def intact(self):
        return [name for name, g in self.g.items() if not g.intact()]


def roots_and_seeds(size, n, seed):
    rng = np.random.RandomState(seed)
    A = T.N_ACTIONS[size]
    depths = rng.randint(1, 9, size=n)
    roots = np.stack([O.scramble(size, rng.randint(A, size=(1, int(d))))[0] for d in depths])
    return roots, [int(s) for s in rng.randint(1 << 30, size=n)]


# (mode, size) -> (constant set, optional-input variant, coverage counters that must be > 0 besides the common
# ones).  Every size meets every constant set and both variants; the aliasing keys run with both variants, and the
# odd path_cap (variant b) meets paths longer than 16 for both sizes.
CASES = {
    ("real", 2): (0, "a", ("path16", "path32")),
    ("real", 3): (1, "b", ()),
    ("colliding", 2): (1, "b", ("overwrite", "self_child", "bounce", "path16")),
    ("colliding", 3): (2, "a", ("overwrite", "self_child", "bounce")),
    ("lastword", 2): (2, "a", ("bounce",)),
    ("lastword", 3): (0, "b", ("path16", "path32")),
    ("firstbyte", 2): (0, "b", ("overwrite", "self_child", "bounce", "path16", "path32")),
    ("firstbyte", 3): (2, "a", ("overwrite", "self_child", "bounce")),
}
COMMON = ("refound", "solved", "budget")


def cosimulate(size, mode, consts, variant, n=B, seed=0):
    """Runs NUM_SIM simulations of n trees on the device and on the oracle, comparing after every call."""
    cpuct, vl, vmin = consts
    A, S = T.N_ACTIONS[size], T.N_STICKERS[size]
    path_cap = 8 * (NUM_SIM + 1) + (1 if variant == "b" else 0)
    M = NUM_SIM + 1
    roots, seeds = roots_and_seeds(size, n, 1000 * size + seed)
    active = np.ones(n, np.uint8)
    active[[i for i in INACTIVE if i < n]] = 0
    ora = OracleBatch(size, mode, consts, roots, active, seeds, M)
    d = DeviceTrees(size, n, M, path_cap, path_cap, with_counter=(variant == "a"))
    d.upload(root_state=roots, root_key=ora.key(roots), active=active,
             rand_table=BatchedMCTS.draw_table(seeds, A, path_cap).numpy())
    inactive0 = np.flatnonzero(active == 0)
    want_active = np.zeros(NUM_SIM, np.int32)
    for sim in range(NUM_SIM):
        # ---- traverse
        assert d.traverse(cpuct, vl) == 0, _lib.load().cube_last_error()
        plen, leaf = ora.traverse()
        torch.cuda.synchronize()
        if variant == "a":
            assert int(d.host("sim_counter")[0]) == sim
        assert int(d.host("flags")[0]) == 0, sim
        got_len = d.host("path_len")
        assert (got_len == plen).all(), (sim, np.flatnonzero(got_len != plen)[:8])
        pn, pa = d.host("path_node"), d.host("path_action")
        for i in np.flatnonzero(ora.active):
            slots, acts = ora.expected_path(i)
            assert pn[i, :plen[i]].tolist() == slots and pa[i, :plen[i]].tolist() == acts, (sim, i)
        got_leaf = d.host("leaf_state")
        assert (got_leaf == leaf).all(), (sim, np.flatnonzero((got_leaf != leaf).any(1))[:8])
        draws = np.array([t.rng.n for t in ora.trees], np.int32)
        assert (d.host("rand_ptr") == draws).all(), sim
        assert (d.host("L") == ora.E["L"]).all(), sim
        # ---- expand + back-up
        was_active = ora.active.copy()
        leaf_keys, child_keys, done, value, policy, solved = ora.update(sim, got_leaf)
        d.upload(leaf_key=leaf_keys, child_key_new=child_keys, child_done_new=done, value=value, policy=policy)
        assert d.update(vmin, sim) == 0, _lib.load().cube_last_error()
        torch.cuda.synchronize()
        check_store(d, ora, sim)
        assert (d.host("active") == ora.active).all(), sim
        out, n_act, n_sims = d.host("actions_out"), d.host("n_actions"), d.host("n_sims")
        for i, acts in solved.items():
            assert out[i, :len(acts)].tolist() == acts and (out[i, len(acts):] == -1).all(), (sim, i)
            assert n_act[i] == len(acts) and n_sims[i] == sim + 1, (sim, i)
        still = np.flatnonzero(ora.active == 1)
        assert (n_act[still] == 0).all() and (n_sims[still] == -7).all() and (out[still] == -1).all()
        assert (n_act[inactive0] == 0).all() and (n_sims[inactive0] == -7).all()
        if variant == "a":
            want_active[sim] = ora.active.sum()
            assert (d.host("n_active") == want_active).all(), sim
        assert (got_len[was_active == 0] == 0).all()
        bad = d.intact()
        assert not bad, (sim, bad)
        if not ora.active.any():
            break
    for i in range(n):
        ora.rebuild(i)
    check_store(d, ora, "final")
    assert ora.cov["longest"] < path_cap // 4                  # the oracle never came near path_cap
    return ora.cov


def check_store(d, ora, sim):
    E = ora.E
    assert (d.host("n_nodes") == E["n_nodes"]).all(), sim
    for name in ("node_key", "child_key", "child_done", "N", "L", "child_slot"):
        got = d.host(name)
        ok = (got == E[name]).reshape(got.shape[0], -1).all(1)
        assert ok.all(), (sim, name, np.flatnonzero(~ok)[:8])
    for name in ("P", "W"):                                    # float equality (no NaN, no -0.0 here)
        got = d.host(name)
        ok = (got == E[name]).reshape(got.shape[0], -1).all(1)
        assert ok.all(), (sim, name, np.flatnonzero(~ok)[:8])


@pytest.mark.parametrize("mode", ("real", "colliding", "lastword", "firstbyte"))
@pytest.mark.parametrize("size", SIZES)
def test_tree_kernels_follow_the_oracle_tree(size, mode):
    """B = 300 trees (three blocks, a ragged last warp and block, trees inactive from the start), roots 1..8 moves
    deep, 40 simulations: after every traversal and every update the device agrees with the oracle's trees.
    Variant a is BatchedMCTS's call (sim_counter from -1, n_active, path_cap a multiple of 4); variant b passes
    sim_counter = n_active = NULL, the simulation index by value and an odd path_cap (the back-up's byte loads)."""
    ci, variant, targets = CASES[(mode, size)]
    cov = cosimulate(size, mode, CONSTS[ci], variant)
    print("coverage", size, mode, CONSTS[ci], variant, cov)
    for name in COMMON + targets:
        assert cov[name] > 0, (name, cov)


def _device_sims(size, d, consts, n_sims, roots, sim_index=True):
    """n_sims simulations on the device alone, keys / values / policies as in the co-simulation (real keys)."""
    cpuct, vl, vmin = consts
    key = make_key("real", size)
    for sim in range(n_sims):
        assert d.traverse(cpuct, vl) == 0
        leaf = d.host("leaf_state")
        children, done = O.expand(size, leaf)
        value, policy = value_policy(key(leaf), T.N_ACTIONS[size])
        d.upload(leaf_key=key(leaf), child_key_new=key(children.reshape(-1, children.shape[-1])), child_done_new=done,
                 value=value, policy=policy)
        assert d.update(vmin, sim) == 0
    torch.cuda.synchronize()


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("case", ("path_cap", "rand_cap", "n_slots", "bad_action"))
def test_capacity_flags_stay_inside_the_buffers(size, case):
    """Each capacity flag of the tree store is raised, and its error path writes nothing outside the caller's
    arrays: 1 path_cap too small, 2 rand_table with too few draws, 4 fewer node slots than simulations + 1,
    8 a pre-drawn action >= A (taken as 0)."""
    A = T.N_ACTIONS[size]
    n, n_sims = 140, 12
    roots, seeds = roots_and_seeds(size, n, 77 + size)
    roots[:] = O.scramble(size, np.random.RandomState(size).randint(A, size=(n, 8)))      # nothing solves early
    path_cap, rand_cap, n_slots = 8 * (n_sims + 1), 8 * (n_sims + 1), n_sims + 1
    if case == "path_cap":
        path_cap = 2
    elif case == "rand_cap":
        rand_cap = 1
    elif case == "n_slots":
        n_slots = 4
    d = DeviceTrees(size, n, n_slots, path_cap, rand_cap, with_counter=True)
    table = BatchedMCTS.draw_table(seeds, A, rand_cap).numpy()
    if case == "bad_action":
        table[::3, 1] = 200
    d.upload(root_state=roots, root_key=real_key(size, roots), active=np.ones(n, np.uint8), rand_table=table)
    _device_sims(size, d, CONSTS[0], n_sims, roots)
    flag = {"path_cap": 1, "rand_cap": 2, "n_slots": 4, "bad_action": 8}[case]
    assert int(d.host("flags")[0]) & flag, int(d.host("flags")[0])
    assert d.intact() == []
    assert (d.host("n_nodes") <= n_slots).all() and (d.host("path_len") <= path_cap).all()
    assert (d.host("n_actions") <= path_cap + 1).all()


def test_batched_mcts_raises_on_capacity_errors():
    """BatchedMCTS.run reports a traversal longer than path_cap and a rand_table that runs out as RuntimeError."""
    from oracle.gen_golden import ExactSearchNet
    size, A, n = 3, 12, 64
    roots = O.scramble(size, np.random.RandomState(3).randint(A, size=(n, 6)))
    net = ExactSearchNet(T.STATE_DIM[size], A).to(dev())
    x = torch.from_numpy(roots).to(dev())
    with pytest.raises(RuntimeError, match="capacity exceeded"):         # (its rand_cap follows path_cap: flags 1 | 2)
        BatchedMCTS(net, size, num_sim=20, path_cap=2).run(x, seeds=list(range(n)))
    with pytest.raises(RuntimeError, match="flags=2:"):
        BatchedMCTS(net, size, num_sim=20).run(x, rand_table=BatchedMCTS.draw_table(range(n), A, 1))
