"""Batched greedy roll-outs: the reference's validation / test loops
(train.py:167-198 `validation`, test.py:103-158 `trial` without MCTS) for many cubes at once.

Reference loop, per cube:  state = env.reset(seed, k);  for t in 1..max_timesteps:
action = model.get_action(state[, pre_action]);  state, reward, done, _ = env.step(action);
stop at the first `done`.  Here every (scramble depth, cube) pair is one row of a batch: the
scrambles run in one fused launch (shallower rows are padded with the no-op action index 12),
and each time step is one encode (K3), one forward of the caller's net and one step (K2).
Rows that are done keep receiving the no-op action, so their state stays solved.

Quirk kept from the reference: `done` is only observed after a step, so a cube whose scramble
happens to end solved is not counted until the policy steps back into the solved state.
"""
import numpy as np
import torch

from . import ops

NOOP = 12          # identity row of every move table (include/cube_b200.h)


def reference_scrambles(cube_size, seeds, depths):
    """moves [len(depths) * len(seeds), max(depths)] uint8 (host), row-major over (depth, seed):
    row (d, s) holds np.random.RandomState(seed_s).randint(A, size=d) -- what reset(seed_s, d)
    draws (cube_env.py:61-68) -- padded with the no-op index."""
    a = ops.N_ACTIONS[cube_size]
    depths = list(depths)
    out = np.full((len(depths) * len(seeds), max(depths)), NOOP, dtype=np.uint8)
    for i, d in enumerate(depths):
        for j, s in enumerate(seeds):
            out[i * len(seeds) + j, :d] = np.random.RandomState(int(s)).randint(a, size=d)
    return out


def reference_scrambles_device(cube_size, seeds, depths, device=None):
    """`reference_scrambles` drawn on the device (C ABI cube_moves_from_seeds): reset(seed, d) uses the
    first d draws of the seed's stream, so one row per seed at the largest depth is cut to every depth
    and padded with the no-op index.  uint8 [len(depths) * len(seeds), max(depths)] on the device."""
    depths = list(depths)
    dmax = max(depths)
    if dmax > 128:                                                                     # deeper than K0 draws
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        return torch.from_numpy(reference_scrambles(cube_size, seeds, depths)).to(dev)
    base = ops.moves_from_seeds(cube_size, seeds, dmax, device=device)                  # [S, dmax]
    d = torch.tensor(depths, device=base.device).view(-1, 1, 1)
    k = torch.arange(dmax, device=base.device).view(1, 1, -1)
    rows = torch.where(k < d, base.unsqueeze(0), torch.full_like(base.unsqueeze(0), NOOP))
    return rows.reshape(len(depths) * base.shape[0], dmax).contiguous()


def greedy_actions(policy_logits, pre_action=None):
    """model.get_action for a batch (model.py:47-76): the best action, or the second best when
    the best one is the inverse (a ^ 1) of `pre_action`.  pre_action: int64 [N] with -1 = none."""
    if pre_action is None:
        return policy_logits.argmax(dim=1)
    top2 = policy_logits.topk(2, dim=1).indices
    invalid = torch.where(pre_action >= 0, pre_action ^ 1, torch.full_like(pre_action, -1))
    return torch.where(top2[:, 0] == invalid, top2[:, 1], top2[:, 0])


@torch.no_grad()
def greedy_solve(model, cube_size, moves, max_timesteps=200, mask_inverse=False, obs_dtype=None,
                 model_device=None):
    """Scramble with `moves` ([N, depth] uint8, host or CUDA; NOOP-padded rows allowed), then follow
    the greedy policy of `model` for at most `max_timesteps` steps.  `obs_dtype` defaults to the dtype the model
    computes in (a bfloat16 DeepCube reads the encode kernel's bf16 rows as they are, no `.float()` pass).

    Returns dict(solved bool [N], steps int64 [N] (time step of the first done, 0 = never),
    states uint8 [N, S] final sticker rows).
    """
    if not torch.cuda.is_available():
        raise RuntimeError("rubiks_cube_solver_b200 needs a CUDA device: there is no CPU fallback")
    if not isinstance(moves, torch.Tensor):
        moves = torch.from_numpy(np.ascontiguousarray(moves, dtype=np.uint8))
    dev = moves.device if moves.is_cuda else torch.device("cuda", torch.cuda.current_device())
    moves = moves.to(dev).contiguous()
    mdev = dev if model_device is None else torch.device(model_device)
    from .adi import model_dtype, param_dtype
    if obs_dtype is None:
        obs_dtype = model_dtype(model)
    in_dtype = param_dtype(model)
    n = moves.shape[0]
    states, _, _ = ops.scramble(cube_size, moves, want_flags=False)
    done = torch.zeros(n, dtype=torch.bool, device=dev)
    steps = torch.zeros(n, dtype=torch.int64, device=dev)
    pre = torch.full((n,), -1, dtype=torch.int64, device=dev)
    obs = torch.empty((n,) + ops.STATE_DIM[cube_size], dtype=obs_dtype, device=dev)
    solved = torch.empty(n, dtype=torch.uint8, device=dev)
    reward = torch.empty(n, dtype=torch.float32, device=dev)
    noop = torch.full((n,), NOOP, dtype=torch.int64, device=dev)
    for t in range(1, max_timesteps + 1):
        ops.encode(cube_size, states, dtype=obs_dtype, out=obs)
        x = obs.to(mdev)
        if in_dtype is not None and x.dtype != in_dtype:
            x = x.to(in_dtype)
        _, logits = model(x)
        action = greedy_actions(logits.float().to(dev), pre if mask_inverse else None)
        action = torch.where(done, noop, action)
        ops.step(cube_size, states, action.to(torch.uint8), solved=solved, reward=reward)
        newly = solved.bool() & ~done
        steps = torch.where(newly, torch.full_like(steps, t), steps)
        done |= newly
        pre = action
        if t % 8 == 0 and bool(done.all()):               # one host synchronisation every eight time steps, not every one
            break
    return dict(solved=done, steps=steps, states=states)


def validation(model, cube_size, sample_scramble_count=30, sample_cube_count=10, max_timesteps=200,
               mask_inverse=False, model_device=None):
    """Solve percentage per scramble depth 1..sample_scramble_count with the reference's seeds
    (seed = 10 * cube index, train.py:180): the list `validation` stores in valid_history."""
    seeds = [i * 10 for i in range(sample_cube_count)]
    depths = list(range(1, sample_scramble_count + 1))
    moves = reference_scrambles_device(cube_size, seeds, depths)
    res = greedy_solve(model, cube_size, moves, max_timesteps=max_timesteps, mask_inverse=mask_inverse,
                       model_device=model_device)
    solved = res["solved"].view(len(depths), len(seeds)).float().mean(dim=1) * 100.0
    return [float(x) for x in solved.cpu()]


def optimal_gap(model, seeds, depths, max_timesteps=200, mask_inverse=False, model_device=None):
    """How far the greedy policy's 2x2x2 solutions are from optimal: `validation`'s solve-% curve with the
    solution-length comparison beside it.  Every (depth, seed) cube is scrambled as reset(seed, depth) draws it and
    solved by `greedy_solve`; the exact distance of every scramble comes from the distance table (ops.distance).

    Returns one dict per depth: depth, solved_pct, mean_distance (over all cubes), mean_steps (over the cubes
    greedy solved) and mean_excess (steps - distance over the cubes greedy solved, leaving out scrambles that
    already end solved: greedy counts those only after stepping back, see the module docstring).  A mean over no
    cube is NaN."""
    seeds, depths = [int(s) for s in seeds], [int(d) for d in depths]
    moves = reference_scrambles_device(2, seeds, depths)
    res = greedy_solve(model, 2, moves, max_timesteps=max_timesteps, mask_inverse=mask_inverse,
                       model_device=model_device)
    start, _, _ = ops.scramble(2, moves, want_flags=False)
    shape = (len(depths), len(seeds))
    dist = ops.distance(2, start).cpu().numpy().reshape(shape).astype(np.int64)
    solved = res["solved"].cpu().numpy().reshape(shape)
    steps = res["steps"].cpu().numpy().reshape(shape)

    def mean(x):
        return float(x.mean()) if x.size else float("nan")

    return [dict(depth=d, solved_pct=float(solved[i].mean()) * 100.0, mean_distance=mean(dist[i]),
                 mean_steps=mean(steps[i][solved[i]]),
                 mean_excess=mean((steps[i] - dist[i])[solved[i] & (dist[i] > 0)]))
            for i, d in enumerate(depths)]
