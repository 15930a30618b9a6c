import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from rubiks_cube_solver_b200 import _lib
if os.environ.get("AB_LIB"): _lib.LIB_PATH = os.environ["AB_LIB"]
from rubiks_cube_solver_b200 import ops
dev = torch.device("cuda", 0)
for size, n, d, a in ((2, 16 << 20, 20, 6), (3, 8 << 20, 30, 12)):
    moves = torch.randint(0, a, (n, d), dtype=torch.uint8, device=dev)
    act = torch.randint(0, a, (n,), dtype=torch.uint8, device=dev)
    S = ops.N_STICKERS[size]
    st = torch.empty((n, S), dtype=torch.uint8, device=dev); so = torch.empty(n, dtype=torch.uint8, device=dev); rw = torch.empty(n, dtype=torch.float32, device=dev)
    best = []
    for rep in range(5):
        for _ in range(5): ops.scramble_step(size, moves, act, out=st, solved=so, reward=rw)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(100): ops.scramble_step(size, moves, act, out=st, solved=so, reward=rw)
        e1.record(); torch.cuda.synchronize()
        best.append(e0.elapsed_time(e1) / 100)
    print(os.environ.get("AB_LIB", "tree")[-40:], "size", size, "fused step median %.5f ms" % sorted(best)[2])
