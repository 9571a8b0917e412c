"""ORACLE (test infrastructure, NOT product code) -- import shim that lets the REAL reference
modules under /root/reference be imported in this container, where `minigrid` and
`gymnasium` are not installed.

`install()` registers stand-in `gymnasium*` / `minigrid*` modules in `sys.modules`, backed by
`oracle/minigrid_restated.py`, and puts the reference checkout first on `sys.path`, so that
`import src.custom_envs.register`, `src.scenario_creator.scenario_creator.ScenarioCreator`,
`src.wrappers.*`, `src.ppo.PPO`, `src.fomaml.FOMAML` execute the reference's own code.

Used only by `tests/golden/make_golden.py` (fixture generation); the tests read the fixtures it wrote.
"""
from __future__ import annotations

import importlib
import os
import sys
import types

from . import minigrid_restated as mg

REFERENCE_ROOT = os.environ.get("MERLIN_REFERENCE_ROOT", "/root/reference")

_registry: dict = {}


def _register(id, entry_point, **kwargs):
    _registry[id] = (entry_point, kwargs)


def _make(id, **kwargs):
    entry_point, base_kwargs = _registry[id]
    mod_name, cls_name = entry_point.split(":")
    cls = getattr(importlib.import_module(mod_name), cls_name)
    # gym.make also wraps in PassiveEnvChecker + OrderEnforcing: both pass observations,
    # rewards and flags through unchanged, so they are omitted here.
    return cls(**{**base_kwargs, **kwargs})


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "src"))


def install():
    if not reference_available():
        raise FileNotFoundError(f"reference checkout not found at {REFERENCE_ROOT}")

    def module(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    spaces = module("gymnasium.spaces", Discrete=mg.Discrete, Box=mg.BoxSpace, Dict=mg.DictSpace)
    wrappers = module("gymnasium.wrappers", FlattenObservation=mg.FlattenObservation)
    module(
        "gymnasium",
        Env=mg.Env,
        Wrapper=mg.Wrapper,
        ObservationWrapper=mg.ObservationWrapper,
        ActionWrapper=mg.ActionWrapper,
        register=_register,
        make=_make,
        spaces=spaces,
        wrappers=wrappers,
    )
    core = module("minigrid.core")
    core.grid = module("minigrid.core.grid", Grid=mg.Grid)
    core.mission = module("minigrid.core.mission", MissionSpace=mg.MissionSpace)
    core.world_object = module(
        "minigrid.core.world_object",
        WorldObj=mg.WorldObj, Goal=mg.Goal, Wall=mg.Wall, Floor=mg.Floor, Lava=mg.Lava,
        Door=mg.Door, Key=mg.Key, Ball=mg.Ball, Box=mg.Box,
    )
    core.constants = module(
        "minigrid.core.constants",
        OBJECT_TO_IDX=mg.OBJECT_TO_IDX, COLOR_TO_IDX=mg.COLOR_TO_IDX, COLORS=mg.COLORS,
        STATE_TO_IDX=mg.STATE_TO_IDX, DIR_TO_VEC=mg.DIR_TO_VEC, TILE_PIXELS=mg.TILE_PIXELS,
    )
    env_mod = module("minigrid.minigrid_env", MiniGridEnv=mg.MiniGridEnv)
    wr = module(
        "minigrid.wrappers",
        FullyObsWrapper=mg.FullyObsWrapper,
        RGBImgPartialObsWrapper=mg.RGBImgPartialObsWrapper,
        ImgObsWrapper=mg.ImgObsWrapper,
    )
    module("minigrid", core=core, minigrid_env=env_mod, wrappers=wr)

    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    # make sure a previously imported product-side `src` mirror does not shadow the reference
    for name in [n for n in sys.modules if n == "src" or n.startswith("src.")]:
        del sys.modules[name]
    return REFERENCE_ROOT
