#!/usr/bin/env python
"""A/B timing of the 2x2x2 expansion kernels: two builds of libcube_b200.so in one process, alternated.

    python tools/expand2_ab.py OTHER_LIB [--reps 7] [--iters 20]

Times, with CUDA events on reachable states, the calls that run the generic 2x2x2 kernels (expand_kernel<2,*>,
encode_kernel<2,*>):
  - adi_f32:   cube_expand, the children's one-hot rows in f32 (+ solved, reward) at the ADI size, 4 Mi parents
               (the generic kernel expands every parent)
  - codes:     cube_expand_codes (children, child and parent codes, solved) at 65 536 leaves, the batched MCTS call
  - encode:    cube_encode bf16 of 4 Mi + 37 rows (whole tiles through leaf_kernel, the ragged tail through
               encode_kernel) and of 48 rows (encode_kernel alone)
Each repetition runs every workload once per library, the two libraries in alternating order; the per-call median
and the spread over repetitions are printed per library, with the card's name and power limit.  Both libraries'
outputs are compared byte for byte first.  Writes nothing."""
import argparse
import ctypes
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from rubiks_cube_solver_b200 import _lib, ops  # noqa: E402


def bind(path):
    lib = ctypes.CDLL(os.path.abspath(path))
    vp, i64, ci = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int
    lib.cube_expand.argtypes = [ci, vp, i64, vp, vp, vp, ci, ci, vp, vp, vp, vp]
    lib.cube_expand_codes.argtypes = [ci, vp, i64, vp, vp, vp, vp, ci, ci, vp, vp, vp, vp]
    lib.cube_encode.argtypes = [ci, vp, i64, vp, ci, ci, vp]
    return lib


def p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def workloads(dev):
    """name -> (call(lib, stream), output tensors)"""
    gen = torch.Generator(device=dev).manual_seed(0)

    def states(n):
        moves = torch.randint(0, 6, (n, 20), dtype=torch.uint8, device=dev, generator=gen)
        return ops.scramble(2, moves, want_flags=False)[0]

    out = {}
    n = 4 << 20
    s = states(n)
    coh = torch.empty((n, 6, 147), dtype=torch.float32, device=dev)
    so = torch.empty((n, 6), dtype=torch.uint8, device=dev)
    rw = torch.empty((n, 6), dtype=torch.float32, device=dev)
    out["adi_f32"] = (lambda lib, st: lib.cube_expand(2, p(s), n, None, p(coh), None, 1, 0, p(so), p(rw), None, st),
                      (coh, so, rw))
    m = 65536
    sm = states(m)
    ch = torch.empty((m, 6, 24), dtype=torch.uint8, device=dev)
    cc = torch.empty((m, 6, 8), dtype=torch.uint8, device=dev)
    pc = torch.empty((m, 8), dtype=torch.uint8, device=dev)
    sso = torch.empty((m, 6), dtype=torch.uint8, device=dev)
    out["codes"] = (lambda lib, st: lib.cube_expand_codes(2, p(sm), m, p(ch), p(cc), p(pc), None, 2, 0, p(sso), None,
                                                          None, st), (ch, cc, pc, sso))
    for k in (n + 37, 48):
        se = states(k)
        oh = torch.empty((k, 7, 21), dtype=torch.bfloat16, device=dev)
        out["encode_%d" % k] = (lambda lib, st, se=se, oh=oh, k=k: lib.cube_encode(2, p(se), k, p(oh), 0, 0, st), (oh,))
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("other", help="the libcube_b200.so to compare with this tree's")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    libs = {"tree": bind(_lib.LIB_PATH), "other": bind(args.other)}
    st = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    work = workloads(dev)
    for name, (call, outs) in work.items():               # same outputs from both builds
        got = []
        for lib in libs.values():
            for t in outs:
                t.view(torch.uint8).fill_(0xA5)
            rc = call(lib, st)
            assert rc == 0, (name, rc)
            torch.cuda.synchronize()
            got.append([t.clone() for t in outs])
        assert all(torch.equal(a.view(torch.uint8), b.view(torch.uint8)) for a, b in zip(*got)), name
    times = {(w, l): [] for w in work for l in libs}
    order = list(libs)
    for rep in range(args.reps):
        for w, (call, _) in work.items():
            iters = args.iters * (50 if w in ("codes", "encode_48") else 1)
            for l in (order if rep % 2 == 0 else order[::-1]):
                for _ in range(3):
                    call(libs[l], st)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(iters):
                    call(libs[l], st)
                e1.record()
                torch.cuda.synchronize()
                times[w, l].append(e0.elapsed_time(e1) * 1e3 / iters)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True).stdout.strip().splitlines()
    except OSError:
        q = []
    print("card: %s (%s)" % (torch.cuda.get_device_name(dev), q[0] if q else "nvidia-smi unavailable"))
    print("%-14s %-6s %10s %10s %10s   (us per call over %d repetitions)" % ("workload", "lib", "median", "min", "max",
                                                                                args.reps))
    for w in work:
        for l in libs:
            t = np.array(times[w, l])
            print("%-14s %-6s %10.2f %10.2f %10.2f" % (w, l, np.median(t), t.min(), t.max()))
        print("%-14s tree / other median: %.4f" % (w, np.median(times[w, "tree"]) / np.median(times[w, "other"])))


if __name__ == "__main__":
    main()
