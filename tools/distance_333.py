"""Time the 3x3x3 pattern-database kernels (csrc/pattern.cu) on one GPU:

    python tools/distance_333.py [--n 16777216] [--solve-rows 4096] [--out profiles/r04_distance_333.json]

* the build of the three tables (cube_pattern_tables_build: four memsets + 14 + 11 + 11 BFS level launches), CUDA
  events over 3 builds after one warm-up build;
* the bound (cube_distance_bound) over n reachable states (scrambles of depth 0..30, 54 B each: 16 Mi states are
  906 MB, larger than the 126 MB L2, so the rows stream from HBM);
* solve_bounded on seeded scrambles of depth 8, 10, 12 and 14 (np.random.RandomState(seed).randint(12, size=depth),
  seeds 0..solve_rows-1) with a budget far above the default: rows per second, mean and maximum nodes per row, and
  the share proven within the default budget (a row is proven within a budget B exactly when its search needs at
  most B nodes, since a smaller budget runs the same search and stops earlier).

The card's name and power limit are read in the same run and recorded beside the numbers."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from distance_222 import card, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--n", type=int, default=16 * 2 ** 20, help="reachable states for the bound rate")
    ap.add_argument("--solve-rows", type=int, default=4096, help="seeded scrambles per depth for solve_bounded")
    ap.add_argument("--budget", type=int, default=1 << 25, help="per-row node budget of the measuring solve")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_distance_333.json"))
    args = ap.parse_args()
    import ctypes
    import torch
    from rubiks_cube_solver_b200 import _lib, ops, rollout
    if not torch.cuda.is_available():
        sys.exit("distance_333.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    lib = _lib.load()
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    gpu = card(0)

    tables = torch.empty(ops._pattern_bytes(3), dtype=torch.uint8, device=dev)
    build_s = timed(lambda: lib.cube_pattern_tables_build(3, ctypes.c_void_p(tables.data_ptr()), stream), 1, 3)
    assert torch.equal(tables, ops.pattern_tables(dev)), "a timed build differs from the cached tables"
    del tables

    g = torch.Generator(device=dev).manual_seed(1234)
    moves = torch.randint(0, 12, (args.n, 30), dtype=torch.uint8, device=dev, generator=g)
    depth = torch.randint(0, 31, (args.n, 1), device=dev, generator=g)
    moves[torch.arange(30, device=dev)[None, :] >= depth] = 12                     # depths 0..30
    states, _, _ = ops.scramble(3, moves, want_flags=False)
    del moves
    bound_s = timed(lambda: ops.distance_bound(3, states), 3, 20)
    bound = ops.distance_bound(3, states)
    assert bool((bound != 255).all()), "a scrambled row was taken for unreachable"
    mean_bound = float(bound.float().mean())
    del states, bound

    seeds = list(range(args.solve_rows))
    solve = []
    for d in (8, 10, 12, 14):
        start, _, _ = ops.scramble(3, rollout.reference_scrambles_device(3, seeds, [d]), want_flags=False)
        ops.solve_bounded(3, start[:64].contiguous(), max_nodes=args.budget)                  # warm-up
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        _, length, lower, nodes = ops.solve_bounded(3, start, max_nodes=args.budget, want_nodes=True)
        torch.cuda.synchronize()
        sec = time.perf_counter() - t0
        length, nodes = length.cpu(), nodes.cpu()
        proven = length != 255
        solve.append({
            "depth": d, "rows": len(seeds), "s": sec, "rows_per_s": len(seeds) / sec,
            "nodes_per_s": float(nodes.sum()) / sec,
            "mean_nodes": float(nodes.double().mean()), "max_nodes": int(nodes.max()),
            "proven_pct_measuring_budget": float(proven.double().mean()) * 100.0,
            "proven_pct_default_budget": float((proven & (nodes <= ops.SOLVE_BOUNDED_MAX_NODES)).double().mean()) * 100.0,
            "mean_length_proven": float(length[proven].double().mean()) if bool(proven.any()) else None,
            "length_hist": {int(k): int(v) for k, v in zip(*torch.unique(length, return_counts=True))},
            "nodes_quantiles": {q: float(torch.quantile(nodes.double(), q)) for q in (0.5, 0.9, 0.99)},
        })
        print(json.dumps(solve[-1]), flush=True)

    out = {
        "gpu": gpu,
        "table_build_ms": build_s * 1e3,
        "table_bytes": ops._pattern_bytes(3),
        "bound": {"states": args.n, "ms": bound_s * 1e3, "states_per_s": args.n / bound_s, "mean_bound": mean_bound},
        "solve_bounded": {"max_length": 14, "measuring_budget": args.budget,
                          "default_budget": ops.SOLVE_BOUNDED_MAX_NODES, "by_depth": solve},
        "method": "CUDA events around back-to-back calls after warm-up (build 1 + 3, bound 3 + 20); bound rows are "
                  "scrambles of depth 0..30 from torch.randint(seed 1234), 54 B each, larger than L2; solve_bounded: "
                  "host clock around one call per depth ending in a device synchronise, after a 64-row warm-up",
    }
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
