"""CPU-side checks of the boundary: the C-ABI library loads, exports every symbol that
include/cube_b200.h declares, rejects bad arguments before touching CUDA, and the host
package mirrors the reference's interface.  No kernel is launched here."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

import rubiks_cube_solver_b200 as R
from rubiks_cube_solver_b200 import _lib
from rubiks_cube_solver_b200 import dist as cdist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    R.build_library()
    return _lib.load()


def test_header_symbols_exported(lib):
    header = open(os.path.join(ROOT, "include", "cube_b200.h")).read()
    declared = set(re.findall(r"^(?:int|int64_t|const char\*)\s+(cube_\w+)\s*\(", header, flags=re.M))
    assert declared == set(_lib.SYMBOLS)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.cube_abi_version() == 2


def test_argument_errors_without_cuda(lib):
    buf = (ctypes.c_uint8 * 256)()
    base = ctypes.addressof(buf)
    aligned = ctypes.c_void_p((base + 15) & ~15)
    odd = ctypes.c_void_p(((base + 15) & ~15) + 1)
    assert lib.cube_scramble(4, aligned, 1, 1, aligned, None, None, None, None) == _lib.CUBE_ERR_SIZE
    assert b"cube_size" in lib.cube_last_error()
    assert lib.cube_scramble(3, aligned, -1, 1, aligned, None, None, None, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_scramble(3, aligned, 1, 1, None, None, None, None, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_scramble(3, odd, 1, 1, aligned, None, None, None, None) == _lib.CUBE_ERR_ALIGN
    assert lib.cube_step(5, aligned, aligned, 1, None, None, None, None) == _lib.CUBE_ERR_SIZE
    assert lib.cube_encode(3, aligned, 1, aligned, 7, 0, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_encode(3, aligned, 1, aligned, 0, 2, None) == _lib.CUBE_ERR_ARG           # unknown encoding
    assert lib.cube_expand(2, odd, 1, None, None, None, 0, 0, None, None, None, None) == _lib.CUBE_ERR_ALIGN
    assert lib.cube_decode(3, aligned, 2, _lib.ENCODING_REFERENCE, 1, aligned, None) == _lib.CUBE_ERR_SIZE   # lossy: no inverse
    assert lib.cube_decode(3, odd, 2, _lib.ENCODING_EXACT, 1, aligned, None) == _lib.CUBE_ERR_ALIGN
    assert lib.cube_scramble_step(3, aligned, None, 1, 1, aligned, None, None, None, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_scramble_prefixes(3, aligned, 1, 527, aligned, None, None, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_scramble_prefixes_max_depth(3) == 526 and lib.cube_scramble_prefixes_max_depth(2) == 1159
    assert lib.cube_pipeline_reset_host(None, None, 1, None, None, None, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_host_alloc(0, None) == _lib.CUBE_ERR_ARG and lib.cube_host_free(aligned) == _lib.CUBE_ERR_ARG
    one = (ctypes.c_uint64 * 1)(1 << 20)
    assert lib.cube_peer_buffer_bytes(64) == 8 * 32 * 4 + 2 * 8 * 64 * 8 and lib.cube_peer_buffer_bytes(0) == _lib.CUBE_ERR_ARG
    assert lib.cube_peer_allreduce_i64(9, 0, one, aligned, 1, 64, 1, None) == _lib.CUBE_ERR_ARG       # > CUBE_PEER_MAX_RANKS
    assert lib.cube_peer_allreduce_i64(1, 0, one, aligned, 65, 64, 1, None) == _lib.CUBE_ERR_ARG
    assert lib.cube_peer_allreduce_i64(1, 0, one, aligned, 1, 64, 0, None) == _lib.CUBE_ERR_ARG       # epochs start at 1
    assert lib.cube_peer_allreduce_i64(1, 0, (ctypes.c_uint64 * 1)((1 << 20) + 64), aligned, 1, 64, 1, None) == _lib.CUBE_ERR_ALIGN
    with pytest.raises(NotImplementedError):
        _lib.check(_lib.CUBE_ERR_SIZE, "x")
    with pytest.raises(IndexError):
        _lib.check(_lib.CUBE_ERR_ACTION, "x")
    with pytest.raises(ValueError):
        _lib.check(_lib.CUBE_ERR_ALIGN, "x")


def test_float_arrays_alignment_without_cuda(lib):
    """Float and int32 arrays start on 4 bytes and float64 arrays on 8 (include/cube_b200.h), else CUBE_ERR_ALIGN
    before any launch -- on the device such a pointer would be a misaligned access."""
    buf = (ctypes.c_uint8 * 256)()
    base = (ctypes.addressof(buf) + 15) & ~15
    a = ctypes.c_void_p(base)
    off = lambda k: ctypes.c_void_p(base + k)
    for size in (2, 3):
        for k in (1, 2):
            assert lib.cube_expand(size, a, 1, None, None, None, 0, 0, None, off(k), None, None) == _lib.CUBE_ERR_ALIGN
            assert lib.cube_expand_codes(size, a, 1, None, a, None, None, 0, 0, None, off(k), None, None) == _lib.CUBE_ERR_ALIGN
            assert lib.cube_solved(size, a, 1, None, off(k), None, None) == _lib.CUBE_ERR_ALIGN
        # cube_adi_targets(size, child_values, child_solved, parent_values, scramble_count, weight, table_len, n,
        #                  target_value, target_policy, error, stream): one pointer off at a time
        for i, ks in ((3, (1, 2)), (4, (1, 2)), (5, (1, 4)), (8, (1, 2)), (9, (1, 2)), (10, (1, 4))):
            for k in ks:
                args = [size, a, a, a, a, a, 8, 1, a, a, a, None]
                args[i] = off(k)
                assert lib.cube_adi_targets(*args) == _lib.CUBE_ERR_ALIGN, (i, k)
    assert b"float64" in lib.cube_last_error()


def test_mcts_tree_pointers_without_cuda(lib):
    """cube_mcts_traverse / cube_mcts_update check every pointer the kernels dereference before any launch
    (include/cube_b200.h): NULL -> CUBE_ERR_ARG (only sim_counter and n_active may be NULL), and a pointer the
    kernels read as a vector or a word off its boundary -> CUBE_ERR_ALIGN.  Every case here is rejected, so
    nothing reaches the device."""
    from rubiks_cube_solver_b200.mcts_batch import _Tree
    buf = (ctypes.c_uint8 * 4096)()
    base = (ctypes.addressof(buf) + 63) & ~63
    ptrs = [name for name, _ in _Tree._fields_[4:]]
    row_vec = ("P", "W", "N", "L")
    word = ("node_key", "child_key", "root_key", "root_state", "leaf_state", "path_node", "path_action", "n_nodes",
            "rand_ptr", "path_len", "flags", "sim_counter")
    # update(size, tree, leaf_key, child_key_new, child_done_new, value, policy, value_min, sim_index, actions_out,
    #        n_actions, n_sims, n_active, stream)
    upd_required = (2, 3, 4, 5, 6, 9, 10, 11)
    upd_word = (2, 3, 5, 6, 10, 11, 12)

    def tree(**over):
        t = _Tree(3, 9, 36, 36, *[base + 64 * i for i in range(len(ptrs))])
        for name, v in over.items():
            setattr(t, name, v)
        return t

    def traverse(size, t):
        return lib.cube_mcts_traverse(size, ctypes.byref(t), ctypes.c_float(1.0), 150, None)

    def update(size, t, over=None):
        p = [ctypes.c_void_p(base + 2048 + 64 * i) for i in range(10)]
        args = [size, ctypes.byref(t), p[0], p[1], p[2], p[3], p[4], ctypes.c_float(-10.0), 0, p[5], p[6], p[7], p[8], None]
        for i, v in (over or {}).items():
            args[i] = v
        return lib.cube_mcts_update(*args)

    for size in (2, 3):
        for name in ptrs:
            if name == "sim_counter":
                continue
            assert traverse(size, tree(**{name: None})) == _lib.CUBE_ERR_ARG, (size, name)
            assert update(size, tree(**{name: None})) == _lib.CUBE_ERR_ARG, (size, name)
        for i in upd_required:
            assert update(size, tree(), {i: None}) == _lib.CUBE_ERR_ARG, (size, i)
        offsets = {name: (1, 2) for name in word}
        offsets.update({name: (4, 8) if size == 3 else (4,) for name in row_vec})
        offsets["child_slot"] = (1,)
        for name, ks in offsets.items():
            for k in ks:
                t = tree(**{name: getattr(tree(), name) + k})
                assert traverse(size, t) == _lib.CUBE_ERR_ALIGN, (size, name, k)
                assert update(size, t) == _lib.CUBE_ERR_ALIGN, (size, name, k)
        for i in upd_word:
            for k in (1, 2):
                assert update(size, tree(), {i: ctypes.c_void_p(base + 2048 + 64 * 9 + k)}) == _lib.CUBE_ERR_ALIGN, (size, i, k)
        # the counts are still checked first, and an empty batch needs no pointers at all
        assert traverse(size, tree(n_slots=256)) == _lib.CUBE_ERR_ARG
        assert traverse(size, tree(path_cap=0)) == _lib.CUBE_ERR_ARG
        assert traverse(size, tree(n_trees=-1)) == _lib.CUBE_ERR_ARG
        empty = _Tree(0, 9, 36, 36)
        assert traverse(size, empty) == 0
        assert lib.cube_mcts_update(size, ctypes.byref(empty), *([None] * 5), ctypes.c_float(-10.0), 0,
                                    *([None] * 5)) == 0
    assert lib.cube_mcts_update(3, None, *([None] * 5), ctypes.c_float(-10.0), 0, *([None] * 5)) == _lib.CUBE_ERR_ARG
    assert b"cube_mcts_update" in lib.cube_last_error()


def test_generated_cuda_tables_are_current():
    subprocess.check_call([sys.executable, os.path.join(ROOT, "rubiks_cube_solver_b200", "csrc", "gen_tables.py"),
                           "--check"])


def test_product_tables_equal_oracle_tables():
    # two independent restatements of the reference's constants must agree
    import importlib.util
    spec = importlib.util.spec_from_file_location(
        "_gen", os.path.join(ROOT, "rubiks_cube_solver_b200", "csrc", "gen_tables.py"))
    g = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(g)
    from oracle import tables as T
    assert (np.array(g.MOVES_3) == T.MOVE_DEFS_3).all() and (np.array(g.MOVES_2) == T.MOVE_DEFS_2).all()
    corner = T.CORNER_INDS_3[:, 0] * 3 + T.CORNER_INDS_3[:, 1]
    edge = T.EDGE_INDS_3[:, 0] * 2 + T.EDGE_INDS_3[:, 1]
    assert g.CORNER_COL_3[:62] == list(corner) and not any(g.CORNER_COL_3[62:])
    assert g.EDGE_COL_3[:55] == list(edge) and not any(g.EDGE_COL_3[55:])
    code = T.PIECE_INDS_2[:, 0] | (T.PIECE_INDS_2[:, 1] << 4)
    assert g.PIECE_CODE_2[:58] == list(code)
    assert g.CORNER_DEFS_REF == T.CORNER_DEFS_3.tolist() and g.EDGE_DEFS_REF == T.EDGE_DEFS_3.tolist()
    assert g.PIECE_DEFS_2 == T.PIECE_DEFS_2.tolist()


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "rubiks_cube_solver_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), f
                assert "oracle/" not in text.replace("``oracle/``", "").replace("import ``oracle", ""), f


def test_interface_mirrors_reference():
    assert R.get_env_config(2) == ([7, 21], 6) and R.get_env_config(3) == ([20, 24], 12)
    with pytest.raises(NotImplementedError):
        R.get_env_config(4)
    for name in ("reset", "step", "init_state", "sim_state_to_state", "state_to_sim_state",
                 "get_random_samples", "get_target_value", "render", "close_render", "save_video"):
        assert callable(getattr(R.CubeEnv, name))
    import inspect
    assert list(inspect.signature(R.make_env).parameters) == ["device", "cube_size"]
    assert list(inspect.signature(R.CubeEnv.reset).parameters) == ["self", "seed", "scramble_count"]
    assert inspect.signature(R.CubeEnv.reset).parameters["scramble_count"].default == 2
    assert list(inspect.signature(R.CubeEnv.get_random_samples).parameters) == [
        "self", "replay_buffer", "model", "sample_scramble_count", "sample_cube_count", "temperature"]


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    with pytest.raises(RuntimeError):
        R.make_env("cpu", 3)
    with pytest.raises(TypeError):
        R.ops.scramble(3, torch.zeros((4, 3), dtype=torch.uint8))


def test_shard_range_partitions():
    for n in (0, 1, 7, 64, 67108864, 1000003):
        for w in (1, 2, 3, 4, 8):
            spans = [cdist.shard_range(n, r, w) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(w - 1))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1


def _gloo_worker(rank, world, port, out):
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    r, lr, w = cdist.init_from_env(backend="gloo")
    lo, hi = cdist.shard_range(1001, r, w)
    # each rank "solves" the multiples of 7 in its slice
    solved = sum(1 for i in range(lo, hi) if i % 7 == 0)
    counters = torch.tensor([solved, hi - lo, 0, 0], dtype=torch.int64)
    cdist.reduce_counters(counters)
    t = cdist.max_over_ranks(1.0 + r, torch.device("cpu"))
    out.put((r, counters.tolist(), cdist.reward_total(counters), t))
    dist.destroy_process_group()


def test_two_rank_counter_reduction_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    want_solved = sum(1 for i in range(1001) if i % 7 == 0)
    for _, counters, total, t in res:
        assert counters[:2] == [want_solved, 1001]
        assert total == 2 * want_solved - 1001
        assert t == 2.0


def test_rollout_host_helpers():
    import torch
    from rubiks_cube_solver_b200 import rollout
    from oracle import cube_np as O
    m = rollout.reference_scrambles(3, seeds=[0, 10, 20], depths=[1, 4, 7])
    assert m.shape == (9, 7) and m.dtype == np.uint8
    for i, d in enumerate((1, 4, 7)):
        for j, s in enumerate((0, 10, 20)):
            row = m[i * 3 + j]
            assert (row[:d] == O.reference_moves(3, s, d)).all() and (row[d:] == rollout.NOOP).all()
    logits = torch.tensor([[0.1, 0.9, 0.3, 0.2], [0.8, 0.1, 0.7, 0.0], [0.0, 0.2, 0.1, 0.9]])
    assert rollout.greedy_actions(logits).tolist() == [1, 0, 3]
    # best action is the inverse of the previous one -> second best (model.py:60-74)
    pre = torch.tensor([0, 1, -1])
    assert rollout.greedy_actions(logits, pre).tolist() == [2, 2, 3]


def test_numa_binding_helper_is_best_effort():
    """dist.bind_host_to_gpu_node never raises (no GPU / hidden sysfs) and parses sysfs cpu lists."""
    from rubiks_cube_solver_b200 import dist as cdist
    assert cdist._parse_cpulist("0-3,8,10-11\n") == {0, 1, 2, 3, 8, 10, 11}
    assert cdist._parse_cpulist("") == set()
    info = cdist.bind_host_to_gpu_node(0)
    assert isinstance(info, dict) and info.get("numa_node") is None or isinstance(info.get("numa_node"), int)


def test_bench_scaling_modes_and_reference_arm_line():
    """bench.py host logic without a GPU: weak / strong instance counts (SURVEY.md 8d config 3: rank r of R owns
    N / R rows), one `config` object shared by both arms, and the reference arm's JSON line (a tiny sample)."""
    import json
    import subprocess
    import sys
    import bench

    class Args:
        scaling, instances_total, instances_per_gpu = "strong", 64 * 2 ** 20, 8 * 2 ** 20

    assert [bench.instances_per_gpu(Args, w) for w in (1, 2, 4, 8)] == [64 * 2 ** 20 // w for w in (1, 2, 4, 8)]
    Args.scaling = "weak"
    assert [bench.instances_per_gpu(Args, w) for w in (1, 8)] == [8 * 2 ** 20] * 2
    cfg = bench.workload_config(8, 8 * 2 ** 20, "weak")
    assert cfg["instances_total"] == 64 * 2 ** 20 and cfg["depth"] == 30 and cfg["cube_size"] == 3
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--gpus", "8", "--steps", "2",
                          "--warmup", "1", "--ref-seconds", "0.5"], capture_output=True, text=True, timeout=300, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["config"] == cfg and line["n_gpus"] == 8 and line["steps"] == 2
    assert line["value"] > 0 and line["e2e"]["value"] == line["value"] and line["cpu_baseline"]["kind"] == "port"
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["unit"] == "transitions/s" and line["higher_is_better"] is True
    for bad in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        out = subprocess.run([sys.executable, os.path.join(root, "bench.py")] + bad, capture_output=True, text=True,
                             timeout=300, cwd=root)
        assert out.returncode == 2 and "error:" in out.stderr and not out.stdout
