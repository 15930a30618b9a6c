"""Time the exact 2x2x2 distance kernels (csrc/distance.cu) on one GPU:

    python tools/distance_222.py [--n 16777216] [--out profiles/r03_distance_222.json]

* the table build (cube_distance_table_build: two memsets + 14 BFS level launches), CUDA events over 20 builds;
* the lookup (cube_distance) and the optimal solve (cube_solve_optimal) over n reachable states (scrambles of
  depth 0..30, 24 B each: 16 Mi states are 400 MB, larger than the 126 MB L2, so the rows stream from HBM);
* the lookup as a fraction of the HBM bound at 25 B per state (24 in, 1 out) against the peak bench.py uses.

The card's name and power limit are read in the same run and recorded beside the numbers."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card(index):
    """Name, power limit and max SM clock of the GPU (read-only NVML / nvidia-smi queries)."""
    import torch
    info = {"name": torch.cuda.get_device_name(index)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=60)
        watts, mhz = [x.strip() for x in q.stdout.strip().split(",")]
        info.update(power_limit_w=float(watts), max_sm_clock_mhz=float(mhz))
    except Exception as exc:                                            # noqa: BLE001 - reported, not guessed
        info["power_limit_w"] = "not read (%s)" % (exc,)
    return info


def peak_hbm_gbs():
    """The HBM peak bench.py divides by: MEASURED_PEAKS.json when present, else its 6650 GB/s fallback."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    return 6650.0, "bench.py fallback (no MEASURED_PEAKS.json)"


def timed(fn, warmup, iters):
    import torch
    for _ in range(warmup):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / 1e3 / iters


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--n", type=int, default=16 * 2 ** 20, help="reachable states for the lookup / solve rates")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_distance_222.json"))
    args = ap.parse_args()
    import ctypes
    import torch
    from rubiks_cube_solver_b200 import _lib, ops
    if not torch.cuda.is_available():
        sys.exit("distance_222.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    table = torch.empty(3674160, dtype=torch.uint8, device=dev)
    build_s = timed(lambda: lib.cube_distance_table_build(2, ctypes.c_void_p(table.data_ptr()), stream), 3, 20)
    assert torch.equal(table, ops.distance_table(dev)), "a timed build differs from the cached table"

    g = torch.Generator(device=dev).manual_seed(1234)
    moves = torch.randint(0, 6, (args.n, 30), dtype=torch.uint8, device=dev, generator=g)
    depth = torch.randint(0, 31, (args.n, 1), device=dev, generator=g)
    moves[torch.arange(30, device=dev)[None, :] >= depth] = 12                     # depths 0..30
    states, _, _ = ops.scramble(2, moves, want_flags=False)
    del moves
    dist = torch.empty(args.n, dtype=torch.uint8, device=dev)
    lookup_s = timed(lambda: ops.distance(2, states, out=dist), 3, 20)
    solve_s = timed(lambda: ops.solve_optimal(2, states), 1, 5)
    _, length = ops.solve_optimal(2, states)
    assert bool((dist != 255).all()) and torch.equal(length, dist), "solve lengths differ from the lookup"

    peak, peak_src = peak_hbm_gbs()
    lookup_gbs = 25.0 * args.n / lookup_s / 1e9
    out = {
        "gpu": card(0),
        "states": args.n,
        "table_build_ms": build_s * 1e3,
        "lookup": {"ms": lookup_s * 1e3, "states_per_s": args.n / lookup_s, "bytes_per_state": 25,
                   "GBps": lookup_gbs, "hbm_peak_GBps": peak, "hbm_peak_source": peak_src, "hbm_frac": lookup_gbs / peak},
        "solve_optimal": {"ms": solve_s * 1e3, "states_per_s": args.n / solve_s,
                          "mean_length": float(length.float().mean())},
        "method": "CUDA events around back-to-back calls after warm-up (build 3 + 20, lookup 3 + 20, solve 1 + 5); "
                  "rows are scrambles of depth 0..30 from torch.randint(seed 1234), 24 B each, larger than L2",
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
