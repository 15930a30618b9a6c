"""Oracle vs the reference's own outputs: the tables, step-by-step walks and seeded resets that
oracle/gen_golden.py recorded from the reference's code (gym-cube's cube_env.py, assets/py333.py,
utils.py) into tests/golden/."""
import numpy as np
import pytest

from oracle import cube_np as O
from oracle import tables as T
from oracle.scalar_env import ScalarCubeEnv

from conftest import golden


def test_tables_live():
    g = golden("reference_tables.npz")
    assert (g["moveDefs"] == T.MOVE_DEFS_3).all()
    assert (g["corner_pieceDefs"] == T.CORNER_DEFS_3).all() and (g["edge_pieceDefs"] == T.EDGE_DEFS_3).all()
    assert (g["corner_pieceInds"] == T.CORNER_INDS_3).all() and (g["edge_pieceInds"] == T.EDGE_INDS_3).all()
    # corner_hashOP / edge_hashOP: the solved cube's pieces hash to their own slots, orientation 0
    s = g["initState_3"].astype(np.int64)
    assert (g["corner_pieceInds"][s[g["corner_pieceDefs"]] @ T.CORNER_HASH_W] == [[i, 0] for i in range(8)]).all()
    assert (g["edge_pieceInds"][s[g["edge_pieceDefs"]] @ T.EDGE_HASH_W] == [[i, 0] for i in range(12)]).all()
    # moveInds order and get_env_config (utils.py): the env's action names and observation shape
    for size in (2, 3):
        assert list(g["actions_%d" % size]) == T.ACTIONS[size] and len(T.ACTIONS[size]) == T.N_ACTIONS[size]
        assert golden("config1_%d.npz" % size)["onehot"].shape[1:] == T.STATE_DIM[size]
    assert (T.STATE_DIM[2], T.N_ACTIONS[2], T.STATE_DIM[3], T.N_ACTIONS[3]) == ((7, 21), 6, (20, 24), 12)


@pytest.mark.parametrize("size", (2, 3))
def test_random_walks_live(size):
    g = golden("walks_%d.npz" % size)
    moves = g["moves"]
    n, d = moves.shape
    _, trail, flags = O.scramble(size, moves, per_step=True)
    enc = O.encode(size, trail.reshape(n * d, -1)).reshape((n, d) + T.STATE_DIM[size])
    for w in range(n):
        for k in range(d):
            assert (g["stickers"][w, k] == trail[w, k]).all()
            assert (g["onehot"][w, k] == enc[w, k]).all()
            assert g["done"][w, k] == flags[w, k] and g["reward"][w, k] == (1.0 if flags[w, k] else -1.0)
    assert g["done"].any()


@pytest.mark.parametrize("size", (2, 3))
def test_reset_live(size):
    g = golden("config1_%d.npz" % size)
    depth = g["moves"].shape[1]
    for seed in (0, 3, 50, 1023):
        moves = O.reference_moves(size, seed, depth)
        assert (moves == g["moves"][seed]).all()
        final = O.scramble(size, moves[None, :])
        assert (g["stickers"][seed] == final[0]).all()
        assert (g["onehot"][seed] == O.encode(size, final)[0]).all()
    saved = np.random.get_state()                              # the failing reset skips its set_state
    with pytest.raises(UnboundLocalError):
        ScalarCubeEnv(size).reset(seed=0, scramble_count=0)    # cube_env.py:69
    np.random.set_state(saved)
