#!/usr/bin/env python
"""Benchmark of the cube-transition hot path (BASELINE.json metric: cube transitions/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A *step* is one pass of the fused scramble (K1) over one batch: BASELINE.json configs[2],
"3x3x3 batched scramble+step, 64M instances x depth 30, sharded across 8xB200", i.e.
8 Mi instances x depth 30 per GPU (weak scaling: every rank owns one such slice; the only
collective is the int64 counter all-reduce after each step).  Moves are synthetic
(`torch.randint`, seed 1234 + rank) and resident in HBM before the timed region; the
move buffer (252 MB) and the outputs (495 MB) are each larger than the 126 MB L2.

Rank 0 prints ONE JSON line: `value` (device-timed, inputs resident), `e2e` (same metric
through the host-buffer C-ABI pipeline, pinned host buffers, H2D+D2H inside the timed
region), `roofline` for the scramble kernel, `cpu_baseline` (the reference-semantics
per-cube Python env on all host cores, N=1 only), the other BASELINE configs measured
briefly (`other_configs`), `clocks`, and `gpu_launches`.

`--impl reference` times the reference's own CPU implementation of the path: the
reference is pure Python and cannot travel to the GPU box (and does not import without
gym/matplotlib), so this arm runs the in-repo restatement of its per-cube env
(oracle/scalar_env.py, same NumPy calls and Python loops as cube_env.py:71-111) on every
host core.  oracle/ is used here only as the thing the reference arm measures.
"""
import argparse
import json
import multiprocessing as mp
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CUBE_SIZE = 3
DEPTH = 30
N_PER_GPU = 8 * 2 ** 20
WORKLOAD = ("BASELINE configs[2]: 3x3x3 batched scramble+step, depth 30, 8 Mi instances per GPU "
            "(= 64 Mi sharded over 8 GPUs); moves resident in HBM, buffers > L2 (no flush needed)")


# ----------------------------------------------------------------------------- CPU arms
_ENV = None


def _cpu_init(cube_size):
    global _ENV
    from oracle.scalar_env import ScalarCubeEnv
    _ENV = ScalarCubeEnv(cube_size)


def _cpu_task(args):
    """One worker's share of a step, timed INSIDE the worker (dispatch and pickling are not the env's work)."""
    depth, n_cubes, seed = args
    import numpy as np
    env, rng = _ENV, np.random.RandomState(seed)
    solved = 0
    t0 = time.perf_counter()
    for _ in range(n_cubes):
        env.init_state()
        for a in rng.randint(env.action_dim, size=depth):
            _, _, done, _ = env.step(a)
        solved += int(done)
    return n_cubes * depth, solved, time.perf_counter() - t0


def _cpu_adi_task(args):
    """get_random_samples(buf, net, depth, cubes, T) (cube_env.py:177-252) with DeepCube's layer shapes on one core."""
    depth, n_cubes, seed = args
    import numpy as np
    import torch
    torch.set_num_threads(1)
    np.random.seed(seed)
    torch.manual_seed(0)
    nn = torch.nn

    class Net(nn.Module):                                   # model.py:7-29, hidden [1024, 256, 128] (config.yaml)
        def __init__(self):
            super().__init__()
            self.enc = nn.Sequential(nn.Flatten(), nn.Linear(480, 1024), nn.ELU(), nn.Linear(1024, 256), nn.ELU())
            self.pol = nn.Sequential(nn.Linear(256, 128), nn.ELU(), nn.Linear(128, 12))
            self.val = nn.Sequential(nn.Linear(256, 128), nn.ELU(), nn.Linear(128, 1))

        def forward(self, x):
            if x.dim() == 2:
                x = x.unsqueeze(0)
            h = self.enc(x)
            return self.val(h), self.pol(h)

    net, buf = Net(), []
    _ENV.device = torch.device("cpu")
    _ENV.get_random_samples(buf, net, depth, 1, 1.0)        # warm-up
    buf = []
    t0 = time.perf_counter()
    _ENV.get_random_samples(buf, net, depth, n_cubes, 1.0)
    return len(buf), 0, time.perf_counter() - t0


class CpuReferencePool(object):
    """The reference-semantics per-cube Python env (oracle/scalar_env.py) on one process per
    host core.  One `run` = every process scrambles `cubes_per_proc` cubes to `depth`."""

    def __init__(self, cube_size, procs):
        self.procs = procs
        self.pool = mp.get_context("spawn").Pool(procs, initializer=_cpu_init, initargs=(cube_size,))
        self.run(DEPTH if cube_size == 3 else 20, 4)        # imports + first-touch, untimed

    def run(self, depth, cubes_per_proc, seed0=1000, procs=None, task=_cpu_task):
        """All workers run their share at once, each timing its own loop.  Returns (seconds, units) with
        units / seconds = the SUM of the workers' own rates (what the cores deliver together while all are busy;
        robust against one worker starting a few milliseconds late) and units = what they produced together."""
        procs = self.procs if procs is None else procs
        res = self.pool.map(task, [(depth, cubes_per_proc, seed0 + i) for i in range(procs)], chunksize=1)
        units = sum(r[0] for r in res)
        rate = sum(r[0] / r[2] for r in res)
        return units / rate, units

    def close(self):
        self.pool.close()
        self.pool.join()


def host_procs():
    return max(1, min(os.cpu_count() or 1, 256))


def cpu_c_oracle(cube_size, depth, n):
    import numpy as np
    from oracle import cube_c
    moves = np.random.RandomState(0).randint(12 if cube_size == 3 else 6, size=(n, depth)).astype(np.uint8)
    cube_c.set_threads(host_procs())                         # torch / torchrun may have pinned OpenMP to one thread
    cube_c.scramble(cube_size, moves[: n // 8])
    t0 = time.perf_counter()
    cube_c.scramble(cube_size, moves)
    dt = time.perf_counter() - t0
    return n * depth / dt, cube_c.num_threads()


def workload_config(world, n_per_gpu, scaling):
    """The `config` object of the JSON line: identical in both arms (`--impl b200` and `--impl reference`)."""
    return {"workload": WORKLOAD, "cube_size": CUBE_SIZE, "depth": DEPTH, "instances_per_gpu": int(n_per_gpu),
            "instances_total": int(world * n_per_gpu), "scaling": scaling}


def instances_per_gpu(args, world):
    """weak (default): every rank owns 8 Mi instances (64 Mi over 8 GPUs); strong: SURVEY.md 8d config 3 whole,
    64 Mi instances split over the ranks (rank r owns rows [r * N / R, (r + 1) * N / R))."""
    if args.scaling == "strong":
        return args.instances_total // world
    return args.instances_per_gpu


def run_reference_arm(args):
    """K timed steps; each step is a bounded sample of the workload sized so that the whole run
    takes about `--ref-seconds` of wall clock whatever K is.  A step's time is the slowest worker's own
    loop time (all workers run concurrently), so pool dispatch is not billed to the reference's env."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    procs = host_procs()
    pool = CpuReferencePool(CUBE_SIZE, procs)
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    # ~28 k transitions/s/core (BASELINE.md section 2): cubes per process per step for the time budget
    cubes = max(64, int(args.ref_seconds * 28000.0 / DEPTH / (steps + warmup)))
    for i in range(warmup):
        pool.run(DEPTH, cubes, seed0=5000 + 1000 * i)
    t_total, tr_total = 0.0, 0
    for i in range(steps):
        dt, n_tr = pool.run(DEPTH, cubes, seed0=100000 + 1000 * i)
        t_total += dt
        tr_total += n_tr
    pool.close()
    value = tr_total / t_total
    sample = ("%d processes x %d cubes x depth %d per step (3x3x3 per-cube Python env, oracle/scalar_env.py = the "
              "reference's cube_env.py:71-111 restated), %d steps, timed inside the workers" % (procs, cubes, DEPTH, steps))
    world = max(1, args.gpus)
    line = {
        "impl": "reference", "metric": "cube transitions/sec", "value": value, "unit": "transitions/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": 1e3 * t_total / steps,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(world, instances_per_gpu(args, world), args.scaling),
        "cpu_baseline": {"value": value, "unit": "transitions/s", "cores": procs, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "transitions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)
    return 0


def cpu_baselines(size, depth, cubes_per_proc):
    """The CPU numbers BASELINE.md section 3 asks for beside the GPU line, all with the reference-semantics per-cube
    Python env (oracle/scalar_env.py), each a bounded sample: all host cores and one process on the benchmark's
    own workload, 2x2x2 on all cores, ADI get_random_samples states/s on all cores, and the plain-C oracle."""
    procs = host_procs()
    out = {}
    pool = CpuReferencePool(size, procs)
    dt, n_tr = pool.run(depth, cubes_per_proc)
    out["cpu_baseline"] = {
        "value": n_tr / dt, "unit": "transitions/s", "cores": procs, "kind": "port",
        "sample": "%d processes x %d cubes x depth %d = %d transitions of the 3x3x3 per-cube Python env "
                  "(oracle/scalar_env.py, reference semantics cube_env.py:71-111), timed inside the workers" % (
                      procs, cubes_per_proc, depth, n_tr)}
    dt1, n1 = pool.run(depth, max(64, cubes_per_proc // 5), procs=1)
    out["cpu_baseline_single_process"] = {"value": n1 / dt1, "unit": "transitions/s", "cores": 1, "kind": "port",
                                          "sample": "1 process x %d cubes x depth %d (3x3x3)" % (n1 // depth, depth)}
    adi_cubes = 8
    dta, na = pool.run(depth, adi_cubes, task=_cpu_adi_task)
    out["cpu_baseline_adi"] = {"value": na / dta, "unit": "ADI states/s", "cores": procs, "kind": "port",
                               "sample": "%d processes x get_random_samples(buf, net, %d, %d, 1.0), 3x3x3, DeepCube "
                                         "[1024, 256, 128] in float32 on one thread each (cube_env.py:177-252)" % (
                                             procs, depth, adi_cubes)}
    pool.close()
    pool2 = CpuReferencePool(2, procs)
    dt2, n2 = pool2.run(20, max(64, cubes_per_proc // 3))
    pool2.close()
    out["cpu_baseline_2x2x2"] = {"value": n2 / dt2, "unit": "transitions/s", "cores": procs, "kind": "port",
                                 "sample": "%d processes x %d cubes x depth 20 (2x2x2 per-cube Python env)" % (
                                     procs, n2 // 20 // procs)}
    cv, threads = cpu_c_oracle(size, depth, 2 ** 21)
    out["cpu_baseline_c"] = {"value": cv, "unit": "transitions/s", "cores": threads, "kind": "port",
                             "sample": "plain-C oracle (OpenMP), 2 Mi instances x depth 30"}
    return out


# ----------------------------------------------------------------------------- clocks
class ClockSampler(object):
    """Samples SM clock and throttle reasons through NVML while the timed region runs.  The thread is
    started BEFORE the warm-up and only records while `recording` is set, so neither its start-up nor
    an NVML query lands on the (still empty) launch queue at the start of the timed region."""
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index, period=0.003):
        self.samples, self.reasons, self.period, self._stop = [], set(), period, threading.Event()
        self.max_mhz, self._h, self._nv = None, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:                                   # noqa: BLE001 - NVML optional
            self._h = None
        if os.environ.get("CUBE_BENCH_NO_NVML") == "1":      # A/B switch: does sampling perturb the timing?
            self._h = None
        self._t = threading.Thread(target=self._run, daemon=True)
        self.recording = False

    def sample_now(self):
        nv = self._nv
        if self._h is None:
            return
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
            bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
            for b, name in self.REASONS.items():
                if bits & b and name != "gpu_idle":
                    self.reasons.add(name)
        except Exception:                                   # noqa: BLE001
            pass

    def _run(self):
        # The first periodic sample comes one period in: an NVML query right at the start of the timed
        # region stalls the (still empty) launch queue for ~0.1 ms.  bench.py takes one more sample by
        # hand after the last launch, while the GPU is still working through the queued steps.
        while not self._stop.wait(self.period):
            if self.recording:
                self.sample_now()

    def __enter__(self):
        if self._h is not None:
            self._t.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._h is not None:
            self._t.join(timeout=2)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ----------------------------------------------------------------------------- GPU arm
def time_launches(torch, fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e-3              # seconds per launch


def measure_other_configs(torch, ops, adi, dev, peak_gbs):
    """BASELINE configs 2, 4, 5 and the single-step kernel, device-timed (CUDA events), with the
    algorithmic bytes of SURVEY.md section 8d."""
    out = {}
    gen = torch.Generator(device=dev).manual_seed(4321)

    def entry(name, seconds, units, unit_name, alg_bytes):
        gbs = alg_bytes / seconds / 1e9
        out[name] = {"value": units / seconds, "unit": unit_name, "ms": seconds * 1e3,
                     "algorithmic_GBps": gbs, "hbm_frac": gbs / peak_gbs}

    # config 2: 2x2x2 fused scramble, 16 Mi x depth 20
    n, d = 16 * 2 ** 20, 20
    moves = torch.randint(0, 6, (n, d), dtype=torch.uint8, device=dev, generator=gen)
    st = torch.empty((n, 24), dtype=torch.uint8, device=dev)
    so = torch.empty(n, dtype=torch.uint8, device=dev)
    rw = torch.empty(n, dtype=torch.float32, device=dev)
    t = time_launches(torch, lambda: ops.scramble(2, moves, out=st, solved=so, reward=rw), 10)
    entry("config2_2x2_scramble_16Mi_x20", t, n * d, "transitions/s", n * (d + 24 + 1 + 4))
    del moves, st, so, rw

    # K2: one step on resident states (3x3x3 8 Mi, 2x2x2 16 Mi): 2S + 1 + 1 + 4 bytes per transition
    for size, n in ((3, 8 * 2 ** 20), (2, 16 * 2 ** 20)):
        s_ = ops.N_STICKERS[size]
        states = ops.solved_states(size, n, dev)
        act = torch.randint(0, ops.N_ACTIONS[size], (n,), dtype=torch.uint8, device=dev, generator=gen)
        so = torch.empty(n, dtype=torch.uint8, device=dev)
        rw = torch.empty(n, dtype=torch.float32, device=dev)
        t = time_launches(torch, lambda: ops.step(size, states, act, solved=so, reward=rw), 10)
        entry("step_%dx%d_resident_%dMi" % (size, size, n >> 20), t, n, "transitions/s", n * (2 * s_ + 6))
        del states, act, so, rw

    # configs[2] read literally as "scramble, then one step": K1p (8 Mi x depth 30) followed by K2p on the
    # states it produced, 31 transitions per instance, both launches inside the timed region
    n, d = 8 * 2 ** 20, 30
    moves = torch.randint(0, 12, (n, d), dtype=torch.uint8, device=dev, generator=gen)
    act = torch.randint(0, 12, (n,), dtype=torch.uint8, device=dev, generator=gen)
    st = torch.empty((n, 54), dtype=torch.uint8, device=dev)
    so = torch.empty(n, dtype=torch.uint8, device=dev)
    rw = torch.empty(n, dtype=torch.float32, device=dev)

    def scramble_then_step():
        ops.scramble(3, moves, out=st, solved=so, reward=rw)
        ops.step(3, st, act, solved=so, reward=rw)

    t = time_launches(torch, scramble_then_step, 20)
    entry("config3_3x3_scramble_then_step_8Mi", t, n * (d + 1), "transitions/s", n * (d + 54 + 5) + n * (2 * 54 + 6))
    # ... and fused into ONE launch (cube_scramble_step): the state never leaves the registers between the two
    t = time_launches(torch, lambda: ops.scramble_step(3, moves, act, out=st, solved=so, reward=rw), 20)
    entry("config3_3x3_scramble_step_fused_8Mi", t, n * (d + 1), "transitions/s", n * (d + 1 + 54 + 5))
    del moves, act, st, so, rw
    # config 2 with its step, fused: 2x2x2, 16 Mi x (depth 20 + 1)
    n, d = 16 * 2 ** 20, 20
    moves = torch.randint(0, 6, (n, d), dtype=torch.uint8, device=dev, generator=gen)
    act = torch.randint(0, 6, (n,), dtype=torch.uint8, device=dev, generator=gen)
    st = torch.empty((n, 24), dtype=torch.uint8, device=dev)
    so = torch.empty(n, dtype=torch.uint8, device=dev)
    rw = torch.empty(n, dtype=torch.float32, device=dev)
    t = time_launches(torch, lambda: ops.scramble_step(2, moves, act, out=st, solved=so, reward=rw), 10)
    entry("config2_2x2_scramble_step_fused_16Mi", t, n * (d + 1), "transitions/s", n * (d + 1 + 24 + 5))
    del moves, act, st, so, rw

    # config 4: 3x3x3 ADI expansion, 4 Mi parents -> bf16 [N,12,480] + solved + reward
    n = 4 * 2 ** 20
    parents, _, _ = ops.scramble(3, torch.randint(0, 12, (n, 30), dtype=torch.uint8, device=dev, generator=gen),
                                 want_flags=False)
    child = torch.empty((n, 12, 20, 24), dtype=torch.bfloat16, device=dev)
    t = time_launches(torch, lambda: ops.expand(3, parents, dtype=torch.bfloat16, child_onehot=child), 5, warmup=2)
    entry("config4_3x3_adi_expand_4Mi_parents", t, n, "parents/s", n * (54 + 12 * (960 + 1 + 4)))
    out["config4_3x3_adi_expand_4Mi_parents"]["child_transitions_per_s"] = 12 * n / t
    del parents

    # config 4 end to end on the device: 139 810 cubes x 30 scramble prefixes (cube_env.py:187-194:
    # every prefix is a sample) -> 4 194 300 parents -> 12 children + bf16 one-hot each.  ONE launch writes
    # all prefixes cube-major (cube_scramble_prefixes), one launch expands them.
    cubes = n // 30
    adi_moves = torch.randint(0, 12, (cubes, 30), dtype=torch.uint8, device=dev, generator=gen)
    trail = torch.empty((cubes, 30, 54), dtype=torch.uint8, device=dev)

    def adi_batch():
        ops.scramble_prefixes(3, adi_moves, out=trail)
        ops.expand(3, trail.view(-1, 54), dtype=torch.bfloat16, child_onehot=child[: 30 * cubes])

    t = time_launches(torch, adi_batch, 3, warmup=1)
    n_par = 30 * cubes
    entry("config4_3x3_adi_prefixes_plus_expand", t, n_par, "parents/s",
          n_par * (54 + 12 * (960 + 1 + 4)) + cubes * 30 * (1 + 54))
    t = time_launches(torch, lambda: ops.scramble_prefixes(3, adi_moves, out=trail), 5, warmup=2)
    entry("scramble_prefixes_3x3_139810x30", t, n_par, "prefix states/s", cubes * 30 * (1 + 54))
    del child, adi_moves, trail
    torch.cuda.empty_cache()
    out["config4_adi_iteration_4Mi"] = measure_adi_iteration(torch, adi, ops, dev, cubes, out["config4_3x3_adi_expand_4Mi_parents"]["ms"])

    # 2x2x2 ADI shape: 6 children + their bf16 one-hot rows per parent (kernel K3c)
    n = 4 * 2 ** 20
    parents2, _, _ = ops.scramble(2, torch.randint(0, 6, (n, 14), dtype=torch.uint8, device=dev, generator=gen),
                                  want_flags=False)
    child2 = torch.empty((n, 6, 7, 21), dtype=torch.bfloat16, device=dev)
    t = time_launches(torch, lambda: ops.expand(2, parents2, dtype=torch.bfloat16, child_onehot=child2), 5, warmup=2)
    entry("adi_2x2_expand_4Mi_parents", t, n, "parents/s", n * (24 + 6 * (294 + 1 + 4)))
    del parents2, child2

    # sim_state_to_state for a resident batch (cube_encode), 3x3x3 bf16
    n = 4 * 2 ** 20
    st, _, _ = ops.scramble(3, torch.randint(0, 12, (n, 15), dtype=torch.uint8, device=dev, generator=gen),
                            want_flags=False)
    obs = torch.empty((n, 20, 24), dtype=torch.bfloat16, device=dev)
    t = time_launches(torch, lambda: ops.encode(3, st, dtype=torch.bfloat16, out=obs), 5, warmup=2)
    entry("encode_3x3_bf16_4Mi", t, n, "states/s", n * (54 + 960))
    del st, obs

    # config 5: 2x2x2 MCTS leaves, 1 Mi: leaf one-hot bf16 + children stickers + done flags
    n = 2 ** 20
    leaves, _, _ = ops.scramble(2, torch.randint(0, 6, (n, 11), dtype=torch.uint8, device=dev, generator=gen),
                                want_flags=False)
    t = time_launches(torch, lambda: ops.expand(2, leaves, dtype=torch.bfloat16, want_children=True,
                                                want_child_onehot=False, want_parent_onehot=True), 10)
    entry("config5_2x2_mcts_leaf_expand_1Mi", t, n, "leaves/s", n * (24 + 294 + 144 + 6 + 24))   # + reward f32 x6
    out["drop_in_get_random_samples"] = measure_drop_in_adi(torch, dev)
    out["drop_in_env_step_latency"] = measure_drop_in_step(torch, dev)
    out["mcts_2x2_batched_search"] = measure_mcts(torch, dev)
    out["config3_3x3_whole_64Mi_on_one_gpu"] = measure_config3_whole(torch, ops, dev, peak_gbs)
    return out


def measure_config3_whole(torch, ops, dev, peak_gbs):
    """SURVEY.md 8d config 3 as ONE device's job: 64 Mi instances x depth 30 (what `--scaling strong --gpus 1` runs
    as the headline): 2 GB of moves in, 3.6 GB of sticker rows + verdicts out per launch."""
    n, d = 64 * 2 ** 20, 30
    gen = torch.Generator(device=dev).manual_seed(1234)
    moves = torch.randint(0, 12, (n, d), dtype=torch.uint8, device=dev, generator=gen)
    st = torch.empty((n, 54), dtype=torch.uint8, device=dev)
    so = torch.empty(n, dtype=torch.uint8, device=dev)
    rw = torch.empty(n, dtype=torch.float32, device=dev)
    t = time_launches(torch, lambda: ops.scramble(3, moves, out=st, solved=so, reward=rw), 10)
    gbs = n * (d + 54 + 5) / t / 1e9
    return {"value": n * d / t, "unit": "transitions/s", "ms": t * 1e3, "algorithmic_GBps": gbs, "hbm_frac": gbs / peak_gbs,
            "instances": n}


def measure_adi_iteration(torch, adi, ops, dev, cubes, expand_alone_ms):
    """One ADI iteration measured AS an iteration (cube_env.py:177-252: scramble prefixes -> 12 children -> net ->
    targets) at BASELINE config 4's size, 139 810 cubes x 30 = 4 194 300 parents, DeepCube's layer shapes
    ([1024, 256, 128], config.yaml) in bfloat16 reading K3's bf16 buffer directly, phases device-timed."""
    nn = torch.nn

    class Net(nn.Module):
        def __init__(self):
            super().__init__()
            self.enc = nn.Sequential(nn.Flatten(), nn.Linear(480, 1024), nn.ELU(), nn.Linear(1024, 256), nn.ELU())
            self.pol = nn.Sequential(nn.Linear(256, 128), nn.ELU(), nn.Linear(128, 12))
            self.val = nn.Sequential(nn.Linear(256, 128), nn.ELU(), nn.Linear(128, 1))

        def forward(self, x):
            if x.dim() == 2:
                x = x.unsqueeze(0)
            h = self.enc(x)
            return self.val(h), self.pol(h)

    torch.manual_seed(0)
    net = Net().to(dev).to(torch.bfloat16)
    gen = torch.Generator(device=dev).manual_seed(5)
    moves = torch.randint(0, 12, (cubes, 30), dtype=torch.uint8, device=dev, generator=gen)
    adi.generate_samples(3, moves[:4096], net, 1.0)                      # warm-up (cuBLAS heuristics, allocator)
    torch.cuda.synchronize()
    timers = {}
    res = adi.generate_samples(3, moves, net, 1.0, timers=timers)
    del res
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = adi.generate_samples(3, moves, net, 1.0)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    del res
    torch.cuda.empty_cache()
    non_net = timers["prefixes_ms"] + timers["expand_ms"] + timers["targets_ms"]
    p = cubes * 30
    return {"parents": p, "samples_per_s": p / wall, "ms": wall * 1e3, "phases_ms": timers, "non_net_ms": non_net,
            "cube_expand_alone_ms": expand_alone_ms, "non_net_over_expand": non_net / expand_alone_ms,
            "net": "DeepCube [1024, 256, 128] bf16, stock torch (out of scope: model.py)",
            "forward_chunk_parents": adi.DEFAULT_FORWARD_CHUNK,
            "note": "non-net = prefixes (one launch, cube-major) + expansion incl. the parents' one-hot rows + target assembly"}


def measure_drop_in_step(torch, dev):
    """One cube per call through the drop-in CubeEnv (C ABI cube_env_host_step: mapped pinned page, two launches,
    one synchronisation), the way train.py:155 / mcts.py:80 / test.py:123 drive the reference's env."""
    import numpy as np
    from rubiks_cube_solver_b200.env import make_env
    res = {"unit": "us/call"}
    for size in (2, 3):
        env = make_env(dev, size)
        env.reset(seed=1, scramble_count=10)
        acts = np.random.RandomState(0).randint(env.action_dim, size=1050)
        for a in acts[:50]:
            env.step(int(a))
        t0 = time.perf_counter()
        for a in acts[50:]:
            env.step(int(a))
        res["step_%dx%dx%d" % (size, size, size)] = (time.perf_counter() - t0) / 1000 * 1e6
    return res


def measure_mcts(torch, dev):
    """test.py's MCTS branch (test.py:139-147: up to numMCTSSim = 50 simulations per cube, config.yaml:29)
    for 65 536 2x2x2 cubes in lock-step through BatchedMCTS (device tree store, one traversal kernel, one leaf batch and one update kernel per
    simulation), beside the reference-semantics per-cube search (oracle/mcts_ref.py) on one host core.
    Net: DeepCube's 2x2x2 layer shapes (147-512-128-{64-6, 64-1}) with the weights of the reference's
    pretrained/222model.pt (BASELINE config 5's net) when the fixture tests/golden/pin222.npz is present."""
    import random
    import numpy as np
    from rubiks_cube_solver_b200 import mcts_batch, ops
    from oracle import mcts_ref
    from oracle.scalar_env import ScalarCubeEnv

    class Net(torch.nn.Module):
        def __init__(self):
            super().__init__()
            nn = torch.nn
            self.enc = nn.Sequential(nn.Flatten(), nn.Linear(147, 512), nn.ELU(), nn.Linear(512, 128), nn.ELU())
            self.pol = nn.Sequential(nn.Linear(128, 64), nn.ELU(), nn.Linear(64, 6))
            self.val = nn.Sequential(nn.Linear(128, 64), nn.ELU(), nn.Linear(64, 1))

        def forward(self, x):
            if x.dim() == 2:
                x = x.unsqueeze(0)
            h = self.enc(x)
            return self.val(h), self.pol(h)

        def predict(self, x):                                  # model.py:78-91
            v, p = self.forward(torch.tensor(x).float())
            return v.numpy()[0], torch.nn.functional.softmax(p, dim=-1).numpy()[0]

    torch.manual_seed(1)
    net = Net()
    weights = "random init"
    fixture = os.path.join(os.path.dirname(os.path.abspath(__file__)), "tests", "golden", "pin222.npz")
    if os.path.exists(fixture):                                # the weights of the reference's pretrained/222model.pt
        g = np.load(fixture)
        names = {"encoder_net": "enc", "policy_net": "pol", "value_net": "val"}
        net.load_state_dict({names[k[2:].split(".")[0]] + k[2 + len(k[2:].split(".")[0]):]: torch.from_numpy(g[k])
                             for k in g.files if k.startswith("w:")})
        weights = "pretrained/222model.pt (epoch %d, tests/golden/pin222.npz)" % int(g["epoch"])
    gpu_net = Net().to(dev)
    gpu_net.load_state_dict(net.state_dict())
    n_trees, num_sim, depth = 65536, 50, 8
    gen = torch.Generator(device=dev).manual_seed(77)
    roots, _, _ = ops.scramble(2, torch.randint(0, 6, (n_trees, depth), dtype=torch.uint8, device=dev, generator=gen),
                               want_flags=False)
    table = torch.randint(0, 6, (n_trees, 8 * (num_sim + 1)), generator=torch.Generator().manual_seed(3), dtype=torch.uint8)

    def timed_search(model, obs_dtype):
        search = mcts_batch.BatchedMCTS(model, 2, num_sim=num_sim, obs_dtype=obs_dtype)
        search.run(roots[:256], rand_table=table[:256])        # warm-up
        best, res = None, None
        for _ in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = search.run(roots, rand_table=table)
            torch.cuda.synchronize()
            dt_ = time.perf_counter() - t0
            best = dt_ if best is None else min(best, dt_)
        return best, res

    dt, res = timed_search(gpu_net, torch.float32)
    timers = {}
    mcts_batch.BatchedMCTS(gpu_net, 2, num_sim=num_sim).run(roots, rand_table=table, timers=timers)
    import copy
    dt16, res16 = timed_search(copy.deepcopy(gpu_net).to(torch.bfloat16), torch.bfloat16)
    tf32_was = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True           # the caller's choice, like the net's dtype: float32 weights, TF32 products
    try:
        dt_tf32, res_tf32 = timed_search(gpu_net, torch.float32)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = tf32_was
    sims = int(res["n_sims"].sum())
    env = ScalarCubeEnv(2)
    torch.set_num_threads(1)
    cpu_sims, t0 = 0, time.perf_counter()
    with torch.no_grad():
        for i in range(3):
            env.sim_cube = roots[i].cpu().numpy().astype(np.int64)
            env.cube = env._observe(env.sim_cube)
            _, used, _ = mcts_ref.solve(net.predict, env, env.cube, num_sim, random.Random(i))
            cpu_sims += used
    cpu_dt = time.perf_counter() - t0
    return {"simulations_per_s_batched_gpu": sims / dt, "simulations_per_s_reference_semantics_1_core": cpu_sims / cpu_dt,
            "trees": n_trees, "solved": int(res["solved"].sum()), "ms": dt * 1e3, "net_weights": weights,
            "phases_ms_float32_net": timers,
            "bf16_net": {"ms": dt16 * 1e3, "solved": int(res16["solved"].sum()),
                         "simulations_per_s": int(res16["n_sims"].sum()) / dt16,
                         "note": "the same search with the net (and the leaves' one-hot rows) in bfloat16: the float32 "
                                 "net's SIMT GEMMs are two thirds of the float32 search's time"},
            "float32_net_tf32_matmul": {"ms": dt_tf32 * 1e3, "solved": int(res_tf32["solved"].sum()),
                                        "simulations_per_s": int(res_tf32["n_sims"].sum()) / dt_tf32},
            "note": "one simulation = traverse + leaf expansion (6 children, net value/policy) + back-propagation "
                    "(mcts.py:36-130); 65 536 cubes scrambled 8 deep, 50 simulations each"}


def measure_drop_in_adi(torch, dev):
    """The reference's own call -- env.get_random_samples(buf, model, 30, 200, T) (train.py:155,
    config.yaml: 200 cubes x 30 scrambles, 3x3x3, hidden [1024, 256, 128]) -- through the drop-in
    CubeEnv (GPU inside) and through the reference-semantics per-cube env on one host core."""
    import numpy as np
    import rubiks_cube_solver_b200 as R
    from oracle.scalar_env import ScalarCubeEnv

    class Net(torch.nn.Module):                               # DeepCube's layer shapes (model.py:7-29)
        def __init__(self):
            super().__init__()
            nn = torch.nn
            self.enc = nn.Sequential(nn.Flatten(), nn.Linear(480, 1024), nn.ELU(), nn.Linear(1024, 256), nn.ELU())
            self.pol = nn.Sequential(nn.Linear(256, 128), nn.ELU(), nn.Linear(128, 12))
            self.val = nn.Sequential(nn.Linear(256, 128), nn.ELU(), nn.Linear(128, 1))

        def forward(self, x):
            if x.dim() == 2:
                x = x.unsqueeze(0)
            h = self.enc(x)
            return self.val(h), self.pol(h)

    torch.manual_seed(0)
    gpu_net = Net().to(dev)
    env = R.make_env(dev, 3)
    np.random.seed(0)
    env.get_random_samples([], gpu_net, 30, 200, 1.0)        # warm-up
    buf = []
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(3):
        env.get_random_samples(buf, gpu_net, 30, 200, 1.0)
    torch.cuda.synchronize()
    ours = 3 * 6000 / (time.perf_counter() - t0)
    cpu_net = Net()
    cpu_env = ScalarCubeEnv(3, device=torch.device("cpu"))
    torch.set_num_threads(1)
    cpu_env.get_random_samples([], cpu_net, 30, 2, 1.0)
    t0 = time.perf_counter()
    cpu_env.get_random_samples([], cpu_net, 30, 20, 1.0)
    ref = 600 / (time.perf_counter() - t0)
    return {"samples_per_s_drop_in_gpu": ours, "samples_per_s_reference_semantics_1_core": ref,
            "note": "one sample = one scramble prefix with its 12 children evaluated by the net and the ADI target "
                    "(cube_env.py:177-252); 200 cubes x 30 per call; includes building the Python dicts"}


def source_sha16():
    """Fingerprint of the scramble kernel's sources: a profile-derived figure (roofline.traffic) is only quoted
    when it was captured from exactly these sources."""
    import hashlib
    h = hashlib.sha256()
    for f in ("scramble.cu", "cube_threads.cuh", "cube_common.cuh", "cube_tables.cuh", "cube_sched.cuh", "cube_bulk.cuh"):
        with open(os.path.join(ROOT, "rubiks_cube_solver_b200", "csrc", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def measure_e2e(torch, ops, cdist, args, dev, rank, world, n, depth, size, barrier, moves, states, solved):
    """The metric end to end through the host-buffer C ABI (pinned host arrays in, pinned host arrays out, every
    copy inside the timed region), on all ranks at once, max over ranks -- next to the plain-copy ceiling of the
    SAME byte counts on the SAME box measured in the SAME run (every rank copying concurrently), so the line says
    how far the pipeline is from what the bus gives at this N.

    Headline: batched `reset(seed, depth)` (cube_env.py:50-69) = cube_pipeline_reset_host: 4 bytes per cube in
    (the moves are drawn on the device, bit-equal to np.random.RandomState(seed).randint), sticker rows + done
    flags + rewards out.  Beside it: host-supplied moves (round 1's e2e: 30 bytes per cube in), and both without
    the reward array (it is +-1 by `done`)."""
    S = ops.N_STICKERS[size]
    pipe = ops.HostScramblePipeline(size, depth, chunk_instances=args.e2e_chunk, n_stages=3, device=dev)
    h_moves = moves.cpu().pin_memory()
    h_seeds = (torch.arange(n, dtype=torch.int64) + rank * n).to(torch.int32).pin_memory()      # seeds 0 .. world*n-1
    h_states = torch.empty((n, S), dtype=torch.uint8).pin_memory()
    h_solved = torch.empty(n, dtype=torch.uint8).pin_memory()
    h_reward = torch.empty(n, dtype=torch.float32).pin_memory()
    steps = max(2, min(args.steps, args.e2e_steps))

    def timed(fn):
        for _ in range(2):
            fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
        dt = cdist.max_over_ranks((time.perf_counter() - t0) / steps, dev)
        barrier()
        return dt

    d_seeds = torch.empty(n, dtype=torch.int32, device=dev)
    d_reward = torch.empty(n, dtype=torch.float32, device=dev)
    s_out, s_in = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

    def plain_copies(h2d, reward):
        with torch.cuda.stream(s_out):
            h_states.copy_(states, non_blocking=True)
            h_solved.copy_(solved, non_blocking=True)
            if reward:
                h_reward.copy_(d_reward, non_blocking=True)
        with torch.cuda.stream(s_in):
            if h2d == "moves":
                moves.copy_(h_moves, non_blocking=True)
            else:
                d_seeds.copy_(h_seeds, non_blocking=True)
        s_out.synchronize()
        s_in.synchronize()

    variants = {}
    counts = {}
    for name, fn, h2d, reward in (
            ("reset_from_seeds", lambda: counts.__setitem__("seeds", pipe.reset(h_seeds, h_states, h_solved, h_reward)[3]), "seeds", True),
            ("reset_from_seeds_no_reward", lambda: pipe.reset(h_seeds, h_states, h_solved, None, want_reward=False), "seeds", False),
            ("host_moves", lambda: counts.__setitem__("moves", pipe.run(h_moves, h_states, h_solved, h_reward)[3]), "moves", True),
            ("host_moves_no_reward", lambda: pipe.run(h_moves, h_states, h_solved, None, want_reward=False), "moves", False)):
        t = timed(fn)
        c = timed(lambda: plain_copies(h2d, reward))
        variants[name] = {"ms_per_step": t * 1e3, "value": world * n * depth / t, "ceiling_ms": c * 1e3,
                          "frac_of_ceiling": c / t,
                          "h2d_bytes_per_step": n * (depth if h2d == "moves" else 4),
                          "d2h_bytes_per_step": n * (S + 1 + (4 if reward else 0))}
    # parity of what came back through the pipeline (host moves ran last: h_states holds its rows)
    counters = ops.new_counters(dev)
    moves.copy_(h_moves)
    ref_states, ref_solved, _ = ops.scramble(size, moves, counters=counters)
    assert bool((h_states[:4096] == ref_states[:4096].cpu()).all()) and counts["moves"] == int(counters[0])
    seeded = ops.scramble(size, ops.moves_from_seeds(size, h_seeds[:4096].to(torch.int64) & 0xffffffff, depth, device=dev))[0]
    pipe.reset(h_seeds[:4096].contiguous(), h_states[:4096])
    assert bool((h_states[:4096] == seeded.cpu()).all())
    pipe.close()
    head = variants["reset_from_seeds"]
    e2e = {"value": head["value"], "unit": "transitions/s", "h2d_bytes_per_step": head["h2d_bytes_per_step"],
           "d2h_bytes_per_step": head["d2h_bytes_per_step"], "ms_per_step": head["ms_per_step"], "steps": steps,
           "ceiling_ms": head["ceiling_ms"], "frac_of_ceiling": head["frac_of_ceiling"],
           "ceiling": "plain pinned D2H of the outputs || H2D of the inputs, same byte counts, all %d ranks at once, max over ranks" % world,
           "api": "cube_pipeline_reset_host (C ABI) via ops.HostScramblePipeline.reset: batched reset(seed, %d), pinned host buffers" % depth,
           "variants": variants}
    return e2e


def replay_own_rows(torch, ops, dev, size, moves, states, solved, reward, rank, n_check=4096):
    """After the timed region every rank replays rows of ITS OWN slice through the plain-C oracle (the first half
    of the sample from the head of the slice, the rest random) and demands byte equality."""
    import numpy as np
    from oracle import cube_c
    n = moves.shape[0]
    half = min(n, n_check // 2)
    idx = np.unique(np.concatenate((np.arange(half), np.random.RandomState(100 + rank).randint(n, size=n_check - half))))
    idx_t = torch.from_numpy(idx).to(dev)
    want, ws, wr, _ = cube_c.scramble(size, moves[idx_t].cpu().numpy())
    ok = bool((states[idx_t].cpu().numpy() == want).all()) and bool((solved[idx_t].cpu().numpy().astype(bool) == ws).all()) \
        and bool((reward[idx_t].cpu().numpy() == wr).all())
    return ok, int(idx.size)


DUMP_ROWS = 1 << 16


def dump_outputs(path, torch, states, solved, reward, counters):
    """`--dump-outputs DIR`: what the last timed step handed its caller, as float32 / float64 .npy files, so two
    builds can be compared output for output.  The per-cube outputs are a fixed sample of DUMP_ROWS rows (seeded,
    sorted; every row when there are no more), 15 MB at 8 Mi instances; `rows` holds their indices and `counters`
    the step's exact [solved, produced] totals over all rows (over all ranks when N > 1)."""
    import numpy as np
    n = states.shape[0]
    rows = np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.RandomState(0).choice(n, DUMP_ROWS, replace=False))
    idx = torch.from_numpy(rows).to(states.device)
    out = {"rows": rows.astype(np.float64), "states": states[idx].float().cpu().numpy(),
           "solved": solved[idx].float().cpu().numpy(), "reward": reward[idx].float().cpu().numpy(),
           "counters": counters[:2].double().cpu().numpy()}
    os.makedirs(path, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), a)


def run_b200_arm(args):
    import torch
    import rubiks_cube_solver_b200 as R
    from rubiks_cube_solver_b200 import adi, ops
    from rubiks_cube_solver_b200 import dist as cdist

    rank, local, world = cdist.init_from_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback on the product path)")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    R.load_library()
    # one process per GPU: keep this rank's host threads and pinned buffers on the GPU's own NUMA node
    numa = cdist.bind_host_to_gpu_node(local) if world > 1 and not args.no_numa_bind else {"numa_node": None}

    n, depth, size = instances_per_gpu(args, world), DEPTH, CUBE_SIZE
    S = ops.N_STICKERS[size]
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    moves = torch.randint(0, 12, (n, depth), dtype=torch.uint8, device=dev, generator=gen)
    states = torch.empty((n, S), dtype=torch.uint8, device=dev)
    solved = torch.empty(n, dtype=torch.uint8, device=dev)
    reward = torch.empty(n, dtype=torch.float32, device=dev)
    # The path's only collective (north star: "NCCL used only for the final solved-count and reward
    # reductions"): every step adds into its own pre-zeroed int64[4] counter row, and ONE SUM all-reduce
    # over the rows of the timed steps closes the timed region, so every step's global solved / produced
    # counts come out exact while the main stream carries nothing but the scramble kernels (consecutive
    # launches chain through programmatic dependent launch).  `--reduce-every-step` issues an asynchronous
    # all-reduce per step instead (measured: 5 % slower at 8 GPUs, NCCL's kernel has to squeeze in between
    # persistent CTAs that fill every SM).
    n_rows = max(3, args.warmup) + args.steps + 8
    cbuf = torch.zeros((n_rows, 4), dtype=torch.int64, device=dev)
    pending = []
    state = {"i": 0, "reduced": 0}
    # the closing all-reduce: one small kernel per rank over NVLink peer memory (csrc/peer.cu) instead of an
    # ncclAllReduce of the same few hundred bytes -- the collective's cost is latency only
    peer, collective = None, "none" if world == 1 else "nccl"
    if world > 1 and args.collective == "peer" and not args.reduce_every_step:
        try:
            peer = cdist.PeerCounters(capacity=4 * n_rows)
            collective = "peer"
        except Exception as e:                            # no symmetric memory on this box: NCCL, and say so
            collective = "nccl (peer exchange unavailable: %s)" % (str(e).splitlines()[0][:120] if str(e) else type(e).__name__)
        flag = torch.tensor([1 if peer is not None else 0], dtype=torch.int64, device=dev)
        torch.distributed.all_reduce(flag, op=torch.distributed.ReduceOp.MIN)
        if int(flag[0]) == 0:                             # all ranks or none
            peer = None
            if collective == "peer":
                collective = "nccl (peer exchange unavailable on another rank)"

    def step():
        k = state["i"]
        state["i"] += 1
        ops.scramble(size, moves, out=states, solved=solved, reward=reward, counters=cbuf[k])
        if args.reduce_every_step:
            h = cdist.reduce_counters_async(cbuf[k])
            if h is not None:
                pending.append(h)

    def drain():
        if args.reduce_every_step:
            for h in pending:
                h.wait()
            del pending[:]
        elif state["i"] > state["reduced"]:
            if peer is not None:
                peer.allreduce_(cbuf[state["reduced"]:state["i"]])
            else:
                cdist.reduce_counters(cbuf[state["reduced"]:state["i"]])
            state["reduced"] = state["i"]
        return cbuf[state["i"] - 1]

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    clocks = ClockSampler(local)
    clocks.__enter__()                                    # thread up and idle before anything is timed
    for _ in range(max(3, args.warmup)):
        step()
    drain()
    barrier()
    e0, e1, ek = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    align = torch.zeros(1, dtype=torch.int32, device=dev)
    barrier()
    # The host-side barrier releases the ranks a few tens of microseconds apart, and the closing all-reduce then
    # waits for the last one: that start skew is not work.  A device-side all-reduce in front of the start event
    # lines the GPUs' streams up (the steps behind it are already queued when it completes).
    cdist.reduce_counters(align)
    clocks.recording = True
    e0.record()
    for _ in range(args.steps):
        step()
    ek.record()                                           # this rank's kernels end here, the collective follows
    totals = drain()                                      # inside the timed region
    e1.record()
    clocks.sample_now()                                   # the queued steps are still running
    barrier()                                             # ... and keep sampling until they are done
    clocks.recording = False
    clocks.__exit__(None, None, None)
    if args.dump_outputs and rank == 0:                   # before the isolated launches below rewrite the buffers
        dump_outputs(args.dump_outputs, torch, states, solved, reward, totals)
    local_step_s = e0.elapsed_time(e1) * 1e-3 / args.steps
    step_s = cdist.max_over_ranks(local_step_s, dev)
    # where a multi-GPU region's time goes: every rank's own kernels (GPUs of one box differ by ~1 %) and what
    # follows them (waiting for the slowest rank + the all-reduce); max / min over ranks
    kern_only_ms = e0.elapsed_time(ek) / args.steps
    tail_ms = ek.elapsed_time(e1)
    spread = {"kernels_ms_per_step_max": cdist.max_over_ranks(kern_only_ms, dev),
              "kernels_ms_per_step_min": -cdist.max_over_ranks(-kern_only_ms, dev),
              "after_last_kernel_ms_max": cdist.max_over_ranks(tail_ms, dev),
              "after_last_kernel_ms_min": -cdist.max_over_ranks(-tail_ms, dev)}
    total_tr = world * n * depth
    value = total_tr / step_s
    solved_total, produced_total = int(totals[0]), int(totals[1])
    assert produced_total == world * n, (produced_total, world * n)

    # parity on THIS rank's slice, every rank (SURVEY.md 8d: sampled replay through the oracle)
    ok, n_replayed = replay_own_rows(torch, ops, dev, size, moves, states, solved, reward, rank)
    bad = torch.tensor([0 if ok else 1, n_replayed, int(solved.sum())], dtype=torch.int64, device=dev)
    cdist.reduce_counters(bad)
    assert int(bad[0]) == 0, "%d rank(s) disagree with the oracle on their own rows" % int(bad[0])
    assert int(bad[2]) == solved_total, (int(bad[2]), solved_total)
    parity = {"rows_replayed_through_oracle": int(bad[1]), "ranks": world, "solved_flags_sum_equals_counters": True}

    # roofline of the dominant kernel: kernel-only launches, CUDA events on the launching stream
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak_gbs, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    else:
        peak_gbs, peak_src = 6650.0, "B200_PROFILING.md fallback (of fallback)"
    # Every timed step is exactly one launch of the dominant kernel on the current stream, so its
    # average duration IS this rank's share of the timed region (CUDA events e0 .. e1 above); a short
    # isolated run (20 launches, nothing else on the device) is reported next to it.
    kern_s = local_step_s
    isolated_s = time_launches(torch, lambda: ops.scramble(size, moves, out=states, solved=solved, reward=reward), 20)
    alg_bytes = n * (depth + S + 1 + 4)
    # DRAM bytes of one launch come from an `ncu --set full` capture (profiles/): quoted only when that capture
    # was taken from exactly the sources this library was built from, and scaled by the instance count
    traffic, traffic_note = None, "no capture of these sources"
    prof = os.path.join(ROOT, "profiles", "scramble3_dram_bytes_per_launch.json")
    if os.path.exists(prof):
        try:
            rec = json.load(open(prof))
            if rec.get("source_sha16") == source_sha16():
                traffic = rec["dram_bytes_per_launch"] * n / rec["instances_per_launch"]
                traffic_note = rec.get("from", "")
            else:
                traffic_note = "profiles/scramble3_dram_bytes_per_launch.json is from other sources (stale): not quoted"
        except Exception:                                   # noqa: BLE001
            traffic = None
    roofline = {"bound": "hbm", "kernel": "scramble_pairs_kernel<3,30,2,plain>", "achieved": alg_bytes / kern_s / 1e9,
                "peak": peak_gbs, "unit": "GB/s", "frac": alg_bytes / kern_s / 1e9 / peak_gbs, "traffic": traffic,
                "traffic_source": traffic_note,
                "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes,
                "kernel_ms": kern_s * 1e3, "kernel_ms_isolated": isolated_s * 1e3,
                "transitions_per_s_kernel_only": n * depth / kern_s,
                "note": "K1p is bound by the shared-memory data pipe (pair-table rows, 87 % of peak) and the ALU pipe "
                        "(PRMT), not by HBM (SURVEY.md 8d, DESIGN.md): the HBM fraction is reported as the contract "
                        "asks; see profiles/"}

    e2e = measure_e2e(torch, ops, cdist, args, dev, rank, world, n, depth, size, barrier, moves, states, solved)

    line = {
        "metric": "cube transitions/sec", "value": value, "unit": "transitions/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": step_s * 1e3, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(world, n, args.scaling),
        "details": {"sm_count": R.load_library().cube_sm_count(),
                    "l2": "inputs (%d MB/GPU) and outputs (%d MB/GPU) exceed the 126 MB L2" % (n * depth >> 20, n * (S + 5) >> 20),
                    "collective": ("int64[4] all-reduce(SUM) per step, asynchronous" if args.reduce_every_step else
                                   "one all-reduce(SUM) of the per-step int64[4] solved/produced counter rows at the end of "
                                   "the timed region; a device-side all-reduce in front of the start event aligns the ranks"),
                    "timed_region_by_rank": spread, "closing_collective": collective, "host_numa_binding_rank0": numa},
        "solved_total": solved_total, "reward_total": 2 * solved_total - produced_total, "parity": parity,
        "e2e": e2e, "roofline": roofline, "gpu_launches": args.steps, "clocks": clocks.summary(),
    }

    if rank == 0 and world == 1:
        if not args.skip_other:
            del moves, states, solved, reward
            torch.cuda.empty_cache()
            line["other_configs"] = measure_other_configs(torch, ops, adi, dev, peak_gbs)
        if not args.skip_cpu:
            line.update(cpu_baselines(size, depth, args.cpu_cubes_per_proc))
    if rank == 0:
        emit(line)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    return 0


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line of the contract, on the process's original stdout."""
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    # Libraries talk on stdout too (NCCL prints its version banner there when NCCL_DEBUG is set):
    # keep a private handle on the real stdout for the JSON line and point fd 1 at stderr.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=("b200", "reference"), default="b200")
    ap.add_argument("--instances-per-gpu", type=int, default=N_PER_GPU)
    ap.add_argument("--scaling", choices=("weak", "strong"), default="weak",
                    help="weak: --instances-per-gpu on every rank; strong: --instances-total split over the ranks "
                         "(SURVEY.md 8d config 3 whole: N = 1 runs all 64 Mi instances on one GPU)")
    ap.add_argument("--instances-total", type=int, default=64 * 2 ** 20)
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--e2e-chunk", type=int, default=1 << 19)
    ap.add_argument("--cpu-cubes-per-proc", type=int, default=15000)
    ap.add_argument("--ref-seconds", type=float, default=60.0)
    ap.add_argument("--reduce-every-step", action="store_true")
    ap.add_argument("--collective", choices=("peer", "nccl"), default="peer",
                    help="N > 1: the counters' closing all-reduce as the library's one-kernel exchange over NVLink peer "
                         "memory (cube_peer_allreduce_i64; falls back to nccl when symmetric memory is unavailable) or as ncclAllReduce")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-other", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true", help="N > 1: do not pin each rank to its GPU's NUMA node")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0's slice) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_b200_arm(args)


if __name__ == "__main__":
    sys.exit(main())
