"""Import the reference's own env from /root/reference (TEST INFRASTRUCTURE ONLY).

The reference tree is read-only, exists only in the build container (never on
the GPU box) and does not import as shipped; ``load_reference()`` applies the
four test-only shims of SURVEY.md section 8c (stub gym, stub matplotlib,
``np.int``, stand-in ``assets/py222.py`` -- all under ``oracle/ref_shims/``)
and returns the reference's modules.  Used by ``oracle/gen_golden.py`` and
``oracle/gen_pin222.py``, which record its outputs under ``tests/golden/``.
"""
import importlib
import os
import sys

import numpy as np

REFERENCE_ROOT = os.environ.get("CUBE_REFERENCE_ROOT", "/root/reference")
_SHIMS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_shims")
_REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_loaded = None


def reference_available():
    return os.path.isfile(os.path.join(
        REFERENCE_ROOT, "gym-cube", "gym_cube", "envs", "cube_env.py"))


class Reference(object):
    """Handles to the reference's modules after a shimmed import."""

    def __init__(self, env_mod, gym_cube_mod, cube_env_mod, py333_mod, model_mod, utils_mod):
        self.env = env_mod
        self.gym_cube = gym_cube_mod
        self.cube_env = cube_env_mod
        self.py333 = py333_mod
        self.model = model_mod
        self.utils = utils_mod

    def make_env(self, cube_size, device="cpu"):
        import torch
        return self.env.make_env(torch.device(device), cube_size)


def load_reference():
    global _loaded
    if _loaded is not None:
        return _loaded
    if not reference_available():
        raise FileNotFoundError("reference tree not found at %s" % REFERENCE_ROOT)
    if not hasattr(np, "int"):
        np.int = int                      # py333.py:171,182,238 use np.int
    for p in (_REPO, os.path.join(REFERENCE_ROOT, "gym-cube"), REFERENCE_ROOT, _SHIMS):
        if p in sys.path:
            sys.path.remove(p)
    # shims first (gym, matplotlib, assets/py222); assets/ is a namespace
    # package so it merges with the reference's own assets/ directory.
    sys.path[:0] = [_SHIMS, REFERENCE_ROOT, os.path.join(REFERENCE_ROOT, "gym-cube"), _REPO]
    gym_cube = importlib.import_module("gym_cube")
    importlib.import_module("gym_cube.envs")   # appends envs/ to sys.path (envs/__init__.py:1-4)
    env_mod = importlib.import_module("env")
    cube_env = importlib.import_module("cube_env")
    py333 = importlib.import_module("assets.py333")
    model = importlib.import_module("model")
    utils = importlib.import_module("utils")
    _loaded = Reference(env_mod, gym_cube, cube_env, py333, model, utils)
    return _loaded
